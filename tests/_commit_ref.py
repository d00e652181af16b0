"""Exact CPU reference of the commitment side of libmsgpu: Goldilocks arithmetic on numpy uint64 arrays, the transforms of
ntt.cu written from their definitions, and the MMCS (leaf hashes, node layers with injection, openings) of mmcs.cu.

Independent of oracle/, host/ and csrc/: the field is p = 2^64 - 2^32 + 1 with p3's two-adic generator chain, the
transforms are a textbook iterative radix-2 DFT, and hashing goes through the official `blake3` package. Every function
takes and returns canonical values (< p). Vectorised over whole matrices, so a 2^24-row transform of one column takes
seconds, not minutes."""
import os
from concurrent.futures import ThreadPoolExecutor

import blake3 as _blake3
import numpy as np

P = 2**64 - 2**32 + 1
GENERATOR = 7
ROOT32 = 1753635133440165772  # two_adic_generator(32)

_P = np.uint64(P)
_EPS = np.uint64(2**32 - 1)  # 2^64 mod p
_M32 = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


# ---- Goldilocks on uint64 arrays ---------------------------------------------------------------------------------------
def add(a, b):
    a = np.asarray(a, dtype=np.uint64)
    s = a + np.asarray(b, dtype=np.uint64)
    s = np.where(s < a, s + _EPS, s)  # carry out of 2^64: 2^64 = 2^32 - 1 (mod p), and the sum stays below p
    return np.where(s >= _P, s - _P, s)


def sub(a, b):
    a = np.asarray(a, dtype=np.uint64)
    b = np.asarray(b, dtype=np.uint64)
    d = a - b
    return np.where(a < b, d - _EPS, d)  # borrow: a - b + 2^64 - (2^64 - p)


def neg(a):
    return sub(np.zeros_like(np.asarray(a, dtype=np.uint64)), a)


def mul(a, b):
    """a * b mod p: the 128-bit product from four 32 x 32-bit limb products, then 2^64 = 2^32 - 1 and 2^96 = -1."""
    a = np.asarray(a, dtype=np.uint64)
    b = np.asarray(b, dtype=np.uint64)
    a0, a1 = a & _M32, a >> _S32
    b0, b1 = b & _M32, b >> _S32
    ll, lh, hl, hh = a0 * b0, a0 * b1, a1 * b0, a1 * b1
    mid = (lh & _M32) + (hl & _M32) + (ll >> _S32)  # < 3 * 2^32
    lo = (ll & _M32) | (mid << _S32)
    hi = hh + (lh >> _S32) + (hl >> _S32) + (mid >> _S32)
    hi_hi, hi_lo = hi >> _S32, hi & _M32
    t0 = lo - hi_hi
    t0 = np.where(lo < hi_hi, t0 - _EPS, t0)
    t1 = hi_lo * _EPS
    r = t0 + t1
    r = np.where(r < t1, r + _EPS, r)
    return np.where(r >= _P, r - _P, r)


def inv(x):
    return pow(int(x), P - 2, P)


def two_adic_generator(bits):
    return pow(ROOT32, 1 << (32 - bits), P)


def powers(g, n):
    """[g^0, ..., g^(n-1)] as uint64, by doubling (log n vector multiplications)."""
    out = np.ones(max(n, 1), dtype=np.uint64)
    k = 1
    while k < n:
        m = min(k, n - k)
        out[k:k + m] = mul(out[:m], np.uint64(pow(int(g), k, P)))
        k += m
    return out[:n]


def rev_perm(log_n):
    """rev_perm(L)[i] = i with its L low bits reversed."""
    i = np.arange(1 << log_n, dtype=np.int64)
    r = np.zeros_like(i)
    for b in range(log_n):
        r |= ((i >> b) & 1) << (log_n - 1 - b)
    return r


def _log2(n):
    assert n > 0 and n & (n - 1) == 0, n
    return n.bit_length() - 1


# ---- transforms (rows are the transform axis, columns are independent) -------------------------------------------------
def _butterflies(x, tw):
    """In place: (u, v) <- (u + tw v, u - tw v) over x[:, 0] / x[:, 1] of shape (blocks, 2, half, w)."""
    u, v = x[:, 0], x[:, 1]
    t = mul(v, tw[None, :, None])
    s = add(u, t)
    v[...] = sub(u, t)
    u[...] = s


def _stage(x, tw):
    """One radix-2 stage, split into independent chunks over threads (numpy releases the GIL inside its loops)."""
    blocks, _, half, _ = x.shape
    if blocks * half < (1 << 16):
        return _butterflies(x, tw)
    k = _THREADS
    if blocks >= k:
        parts = [(x[i * blocks // k:(i + 1) * blocks // k], tw) for i in range(k)]
    else:
        parts = [(x[:, :, i * half // k:(i + 1) * half // k], tw[i * half // k:(i + 1) * half // k]) for i in range(k)]
    list(_pool().map(lambda a: _butterflies(*a), parts))


_THREADS = max(1, min(16, os.cpu_count() or 1))
_POOL = []


def _pool():
    if not _POOL:
        _POOL.append(ThreadPoolExecutor(_THREADS))
    return _POOL[0]


def dft(m):
    """dft(f)_k = sum_j f_j w_n^{jk}, natural order in and out: iterative radix-2 decimation in time."""
    m = np.asarray(m, dtype=np.uint64)
    n, w = m.shape
    log_n = _log2(n)
    x = np.ascontiguousarray(m[rev_perm(log_n)])
    if n == 1:
        return x
    tw_all = powers(two_adic_generator(log_n), n // 2)  # w_n^i, i < n/2
    for s in range(1, log_n + 1):
        half = 1 << (s - 1)
        _stage(x.reshape(n >> s, 2, half, w), np.ascontiguousarray(tw_all[:: n >> s][:half]))  # w_{2^s}^i
    return x


def idft(m):
    """The inverse of dft: f_j = n^-1 dft(y)_{(n - j) mod n}."""
    m = np.asarray(m, dtype=np.uint64)
    n = m.shape[0]
    y = dft(m)
    return mul(y[(-np.arange(n)) % n], np.uint64(inv(n)))


def dft_bitrev(m):
    """dft(m).bit_reverse_rows(): row i holds frequency rev(i)."""
    y = dft(m)
    return y[rev_perm(_log2(y.shape[0]))]


def coset_lde_bitrev(m, added_bits, shift=GENERATOR):
    """out[i] = P_c(shift * w_{nB}^{rev(i)}) for the polynomial P_c of degree < n through column c: one zero-padded
    transform of size n * B (B = 2^added_bits) of the coefficients scaled by shift^j."""
    m = np.asarray(m, dtype=np.uint64)
    n, w = m.shape
    coeffs = mul(idft(m), powers(shift, n)[:, None])
    big = np.zeros((n << added_bits, w), dtype=np.uint64)
    big[:n] = coeffs
    return dft_bitrev(big)


def lde_from_shifted_coefficients(coeffs, added_bits):
    """Zero-pad the coefficients to n * B rows, one DFT, bit-reversed storage."""
    coeffs = np.asarray(coeffs, dtype=np.uint64)
    n, w = coeffs.shape
    big = np.zeros((n << added_bits, w), dtype=np.uint64)
    big[:n] = coeffs
    return dft_bitrev(big)


def shifted_quotient_slices(evals, q):
    """evals: nq x d evaluations on the coset GENERATOR * H_{nq}, natural order. out[r][k*d + c] = a_{k*n + r, c} *
    GENERATOR^{-k*n}, with a the coefficients of idft(evals) and n = nq / q: slice k of the quotient, rescaled so that its
    coset LDE is the plain LDE of the output (oracle/cpu_dft.hpp, shifted_quotient_slices)."""
    evals = np.asarray(evals, dtype=np.uint64)
    nq, d = evals.shape
    n = nq // q
    a = idft(evals)
    step = inv(pow(GENERATOR, n, P))
    out = np.empty((n, q * d), dtype=np.uint64)
    for k in range(q):
        out[:, k * d:(k + 1) * d] = mul(a[k * n:(k + 1) * n], np.uint64(pow(step, k, P)))
    return out


# ---- MMCS (BLAKE3, arity 2, cap height 0) --------------------------------------------------------------------------------
def b3(data):
    return _blake3.blake3(data).digest()


def leaf_digests(mats):
    """One digest per row of a height class: BLAKE3 of the rows of all its matrices, concatenated in commit order, as
    little-endian u64. Returns an (h, 32) uint8 array."""
    h = mats[0].shape[0]
    cat = np.ascontiguousarray(np.concatenate([np.asarray(m, dtype=np.uint64).reshape(h, -1) for m in mats], axis=1))
    raw = cat.astype("<u8").tobytes()
    rb = len(raw) // h if h else 0
    return _digests([b3(raw[i * rb:(i + 1) * rb]) for i in range(h)])


def _digests(blist):
    return np.frombuffer(b"".join(blist), dtype=np.uint8).reshape(len(blist), 32).copy()


def node_layers(leaves, inject=None):
    """Digest layers from the leaves up: node i of a layer = BLAKE3(left || right), then BLAKE3(node || inject[len][i]) when a
    class of that height is injected. inject: {height: (height, 32) uint8}. Returns a list of (len, 32) uint8 arrays."""
    inject = inject or {}
    layers = [np.ascontiguousarray(leaves, dtype=np.uint8)]
    while layers[-1].shape[0] > 1:
        prev = layers[-1].tobytes()
        nl = layers[-1].shape[0] // 2
        nodes = [b3(prev[64 * i:64 * i + 64]) for i in range(nl)]
        if nl in inject:
            ij = inject[nl].tobytes()
            nodes = [b3(nodes[i] + ij[32 * i:32 * i + 32]) for i in range(nl)]
        layers.append(_digests(nodes))
    return layers


def class_digests(mats):
    """{height: leaf digests} of the height classes of a commitment; matrices of one height in commit order."""
    by_h = {}
    for m in mats:
        by_h.setdefault(m.shape[0], []).append(m)
    return {h: leaf_digests(g) for h, g in by_h.items()}


def mmcs_commit(mats):
    """MerkleTreeMmcs::commit: all digest layers, leaves first; the root is layers[-1][0]."""
    cls = class_digests(mats)
    top = max(cls)
    return node_layers(cls[top], {h: d for h, d in cls.items() if h != top})


def open_rows(mats, index):
    """The opened rows of open_batch at `index` of the tallest height: matrix m gives row index >> (log max - log h_m)."""
    log_max = _log2(max(m.shape[0] for m in mats))
    rows = [np.asarray(m, dtype=np.uint64)[index >> (log_max - _log2(m.shape[0]))] for m in mats]
    return np.concatenate(rows) if rows else np.zeros(0, dtype=np.uint64)


def open_path(layers, index):
    """The sibling digests of `index`, bottom-up: one per layer below the root. (depth, 32) uint8."""
    return np.stack([layers[l][(index >> l) ^ 1] for l in range(len(layers) - 1)]) if len(layers) > 1 else np.zeros((0, 32), np.uint8)


def open_batch_multi(trees, shifts, indices):
    """msgpu_open_batch_multi's output layout. trees[k] = (mats, layers): mats = the matrices in commit order (an empty list
    for a paths-only tree), layers = the digest layers (None for a rows-only local part). Tree k is opened at
    indices[q] >> shifts[k]; per tree, n_idx rows of the concatenated widths, then n_idx paths, tree after tree."""
    opened, proofs = [], []
    for (mats, layers), s in zip(trees, shifts):
        for ix in indices:
            i = int(ix) >> s
            if mats:
                opened.append(open_rows(mats, i))
            if layers is not None:
                proofs.append(open_path(layers, i))
    o = np.concatenate(opened) if opened else np.zeros(0, dtype=np.uint64)
    p = np.concatenate(proofs) if proofs else np.zeros((0, 32), dtype=np.uint8)
    return o, p
