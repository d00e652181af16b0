"""The NTT tiles of ntt.cu: the power-of-two twiddles they hard-code, and GPU parity at the tile sizes the other NTT tests
do not reach (9-bit tiles in both directions, and the unfused LDE path whose first forward pass is k_ntt_block).

A tile runs radix-16 / radix-16 / rest rounds (DIF) or their mirror image (DIT). Every twiddle of order <= 64 is
two_adic_generator(k) = 2^root_exp(k), k <= 6, applied as a shift; its inverse is 2^(192 - root_exp(k)) since 2^192 = 1."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from tests import _oracle as orc
from tests._naive import P, two_adic_generator

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NTT_CU = os.path.join(ROOT, "multi_stark_b200", "csrc", "ntt.cu")


def _root_exp_source():
    src = open(NTT_CU).read()
    body = re.search(r"constexpr int root_exp\(int logr, bool inv\) \{(.*?)\n\}", src, re.S).group(1)
    exps = {int(k): int(e) for k, e in re.findall(r"logr == (\d+) \? (\d+)", body)}
    inverse = re.search(r"return inv \? \((\d+) - e\) % (\d+) : e;", body)
    return exps, inverse


def test_root_exp_is_the_two_adic_generator():
    exps, inverse = _root_exp_source()
    assert sorted(exps) == [1, 2, 3, 4, 5, 6]
    assert inverse is not None and inverse.groups() == ("192", "192")
    assert pow(2, 96, P) == P - 1 and pow(2, 192, P) == 1
    for k, e in exps.items():
        g = two_adic_generator(k)
        assert pow(2, e, P) == g, k
        assert pow(2, (192 - e) % 192, P) == pow(g, P - 2, P), k
    assert [exps[k] for k in range(1, 7)] == [96, 48, 120, 156, 78, 39]
    # the chain stops at 64: no power of two is a primitive 128th root, so order-128 twiddles stay table multiplications
    assert two_adic_generator(7) not in {pow(2, e, P) for e in range(192)}


def _edge_matrix(rng, rows, cols):
    m = orc.rand_matrix(rng, rows, cols)
    flat = m.reshape(-1)
    flat[:4] = [P - 1, 0, 1, P - 2**32]
    return m


@pytest.fixture(scope="module")
def gpu():
    import multi_stark_b200 as ms
    ctx = ms.GpuContext(0)
    yield ms, ctx
    ctx.close()


# 2^9: one 9-bit tile; 2^18 = 9 + 9 bits, 2^19 = 10 + 9 bits (the fused middle pass of the LDE runs a 9-bit DIT tile)
@pytest.mark.gpu
@pytest.mark.parametrize("log_h,lb,w", [(9, 1, 5), (9, 2, 3), (18, 1, 3), (19, 1, 2), (19, 2, 1)])
def test_coset_lde_nine_bit_tiles(gpu, oracle, log_h, lb, w):
    ms, ctx = gpu
    m = _edge_matrix(np.random.default_rng(900 + log_h + lb), 1 << log_h, w)
    got = ms.GpuDft(ctx).coset_lde_batch_bitrev(m, lb, 7)
    assert np.array_equal(got, orc.coset_lde(oracle, m, lb, 7))


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,w", [(9, 6), (18, 2), (19, 1)])
def test_dft_nine_bit_tiles(gpu, oracle, log_n, w):
    ms, ctx = gpu
    m = _edge_matrix(np.random.default_rng(90 + log_n), 1 << log_n, w)
    got = ms.GpuDft(ctx).dft_batch_bitrev(m)
    assert np.array_equal(got, orc.dft_bitrev(oracle, m))


_UNFUSED = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import multi_stark_b200 as ms
from tests import _oracle as orc
L = orc.lib()
ctx = ms.GpuContext(0)
dft = ms.GpuDft(ctx)
for log_h, lb, w in [(5, 1, 3), (6, 2, 2), (11, 1, 3), (13, 1, 2), (19, 1, 2), (20, 1, 2)]:
    m = orc.rand_matrix(np.random.default_rng(log_h), 1 << log_h, w)
    assert np.array_equal(dft.coset_lde_batch_bitrev(m, lb, 7), orc.coset_lde(L, m, lb, 7)), (log_h, lb, w)
ctx.close()
print("ok")
"""


@pytest.mark.gpu
def test_unfused_coset_lde():
    """MSGPU_LDE_UNFUSED=1 (read once per process) runs the whole inverse transform, then k_ntt_block per coset: its DIT tile
    at 5, 6, 9 and 10 bits."""
    env = dict(os.environ, MSGPU_LDE_UNFUSED="1")
    r = subprocess.run([sys.executable, "-c", _UNFUSED, ROOT], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr
