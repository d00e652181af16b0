"""ONE proof over the ROW SHARDS of every committed matrix (host/rowshard_backend.hpp): every rank holds 1 / N of the rows of
every LDE, so a single tall circuit is proved by all ranks -- column-sharded NTT between two all-to-alls, leaf hashing and
subtrees per rank, stage-2 traces from row blocks, quotient rows with the next rows fetched from another shard, barycentric
sums and reduced openings per shard. The proof must be byte-identical to the single-GPU proof. On a single-GPU box the ranks
share cuda:0 and exchange over gloo (device buffers staged through the host); tools/dist_prove.py runs the same worker over
NCCL with one GPU per rank."""
import pytest

from tests import _oracle as orc
from tests.test_gpu_dist_prove import run_world

pytestmark = pytest.mark.gpu


CASES = [
    # world, kind, log_heights, params
    (2, "u32_add", [10], dict(log_blowup=1, num_queries=20)),                       # q = 1: the quotient domain is one shard
    (4, "u32_add", [11], dict(log_blowup=1, num_queries=15)),                       # two shards span it: next rows fetched
    (2, "u32_add", [9], dict(log_blowup=2, num_queries=12, log_final_poly_len=1)),
    (4, "multi:3", [12, 10, 11], dict(log_blowup=1, num_queries=10)),               # three heights + the byte table in one MMCS
    (2, "wide:16", [9], dict(log_blowup=2, num_queries=10)),                        # lookup-free, quotient degree 2, narrow stage 2
    (4, "wide:16", [10], dict(log_blowup=2, num_queries=10)),
    (4, "wide:16", [10], dict(log_blowup=1, num_queries=10)),                       # q = B: every shard holds quotient rows
    (2, "fib", [8], dict(log_blowup=2, num_queries=8)),                             # 3 columns >= 2 ranks: next-row constraints
    (2, "mixed", [9, 8], dict(log_blowup=2, num_queries=12)),
    (2, "u32_add", [10], dict(log_blowup=1, num_queries=10, commit_pow_bits=2, query_pow_bits=2)),  # host-loop FRI on the owner
    (2, "wide:16", [8], dict(log_blowup=2, num_queries=20)),
    (4, "wide:8", [8], dict(log_blowup=2, num_queries=20)),                         # the least height split over 4 ranks
    (2, "wide:64", [10], dict(log_blowup=1, num_queries=20)),
    (2, "wide:256", [10], dict(log_blowup=2, num_queries=20)),                      # BASELINE configs[2]'s width
]


@pytest.mark.parametrize("world,kind,log_heights,params", CASES)
def test_rowsharded_proof_is_byte_identical(tmp_path, oracle, world, kind, log_heights, params):
    proofs, single, infos = run_world(tmp_path, world, kind, log_heights, "rowshard", params)
    for r in range(world):
        assert proofs[r] == single, "rank %d's proof differs from the single-GPU proof" % r
    assert all(i["launches"] > 0 for i in infos)
    # exchanged device bytes stay a fraction of the committed data: nothing of the size of a matrix is gathered on one rank
    assert all(i["bytes_dev"] > 0 for i in infos)


@pytest.mark.parametrize("world,log_rows,width,lb", [(4, 8, 200, 1), (2, 7, 7, 3), (4, 12, 130, 1)])
def test_rowsharded_commit_of_any_width(tmp_path, world, log_rows, width, lb):
    """RowShardProver.commit of one matrix whose width need not be a wide:W circuit's: every rank's root equals the single-GPU
    `Pcs::commit` of the whole matrix"""
    roots, single, infos = run_world(tmp_path, world, "commit:%d" % width, [log_rows], "rowshard", dict(log_blowup=lb))
    for r in range(world):
        assert roots[r] == single, "rank %d's root differs from the single-GPU commitment" % r
    assert all(i["rows"] == (1 << log_rows) // world for i in infos), "the matrix was not split by rows"
    assert all(i["bytes_dev"] > 0 for i in infos)
