// ONE proof over the ROW SHARDS of every committed matrix (SURVEY 8e carried past the commitment: partitioning B for every
// circuit, so that a single tall circuit no longer pins one GPU).
//
// One process per GPU; every rank runs the SAME prove() driver (prover.hpp) with a replicated Fiat-Shamir transcript over this
// backend. Rank d of N holds, of every committed LDE of height H, the stored rows [d H / N, (d + 1) H / N) -- all columns -- in
// bit-reversed row-major storage. What moves, and why it has to:
//   * Pcs::commit of a wide enough matrix (width >= N): each rank uploads its natural-order ROW block of the evaluations
//     (1 / N of the PCIe traffic), an all-to-all turns row blocks into COLUMN blocks (the NTT is column-local), each rank extends
//     its columns, a second all-to-all turns the LDE's column blocks into row shards. Narrow matrices (stage-2 traces of
//     lookup-free circuits, quotient matrices, byte tables) are made whole on every rank instead (all-gather of the row blocks,
//     then the full LDE everywhere): 2 to 4 columns cannot be split over 8 ranks, and they are a few percent of the work.
//   * MMCS: every rank hashes the leaves of its rows and builds its subtree (shorter matrices are injected inside it: layer
//     length h of the tree is rows [d h / N, ...) of that matrix on rank d); the N subtree roots (32 bytes each) are
//     all-gathered and the top log2 N levels built on every rank. Root and openings are those of a single-GPU commit.
//   * stage-2 (logUp) traces: row-local messages and inverses on the natural-order row block each rank kept from the upload; the
//     running sum needs the ranks' totals (16 bytes each, all-gathered) as an offset.
//   * quotient: every rank evaluates the quotient-domain rows it holds (the first n q stored rows of the LDEs). The NEXT trace row
//     of stored row j is stored row rev(rev(j) + q): one trace step changes the LOW bits of the natural index, i.e. the shard --
//     all next rows of shard d live in shard rev((rev(d) + q) mod N'), which is fetched once (a permutation, one all-to-all
//     call per matrix); the evaluations (16 bytes per row) are all-gathered and every rank finishes the 2q-column quotient LDE.
//   * Pcs::open: barycentric sums over the rows a rank holds, added over the ranks (a few KB); reduced openings row-local, the
//     shards (16 bytes per LDE row) added into the FRI owner's vectors; the FRI fold-and-commit rounds run on the owner with the
//     transcript on the device and ONE broadcast of roots and final polynomial (the other ranks replay the transcript); query
//     rows and lower sibling paths come from the rank that holds the row, the top log2 N siblings from the replicated top tree.
// With peer memory (msh_comm::peer_memory, csrc/peer.cu) the exchanges of a commitment are kernels of this library over NVLink:
// row blocks are written straight into the owners' column blocks (remote stores), row shards are assembled from the peers'
// LDE column blocks (remote loads), the subtree roots are stored into every peer's window, and the only synchronisation is a
// flag barrier in peer memory (no host round trip, no NCCL launch): three barriers per commitment.
// Nothing of the size of a committed matrix is ever gathered on one rank. The proof is byte-identical to the single-GPU proof
// (tests/test_gpu_rowshard.py).
#pragma once
#include "dist_backend.hpp"

namespace msh {

// A block of the symmetric peer heap: the same (segment, offset) on every rank.
struct SymBlock {
    uint32_t seg = 0;
    uint64_t off = 0;
    bool live = false;
};

// Pcs::ProverData of a row-sharded commitment.
struct RowShardHandle : PcsHandle {
    int n_shards = 1, shard = 0;
    std::vector<std::pair<size_t, size_t>> shapes;  // (GLOBAL LDE height, width), commit order
    std::vector<uint64_t*> views;                   // this rank's rows of matrix i: shapes[i].first / n_shards rows
    std::vector<bool> whole;                        // views[i] points into the WHOLE LDE (every rank has every row)
    std::vector<DevBuf> owned;                      // device buffers behind the views (shard buffers or whole LDEs)
    // (pointer, width) of the column blocks a view is still to be assembled from (peer memory: the shard is written by the
    // pass that hashes it); empty once the commitment is built
    std::vector<std::vector<std::pair<const uint64_t*, uint64_t>>> pending;
    PdataPtr local;                                 // MMCS over the views: leaf digests + subtree of this rank's rows
    PdataPtr top;                                   // the top log2(n_shards) levels over the subtree roots
    size_t num_matrices() const override { return shapes.size(); }
    size_t matrix_height(size_t i) const override { return shapes[i].first; }
    size_t matrix_width(size_t i) const override { return shapes[i].second; }
    size_t shard_rows(size_t i) const { return shapes[i].first / (size_t)n_shards; }
    // rows of shard `e` of matrix i when the whole LDE is here
    uint64_t* whole_rows_of(size_t i, int e) const { return views[i] + ((ptrdiff_t)e - shard) * (ptrdiff_t)(shard_rows(i) * shapes[i].second); }
};

inline unsigned rs_rev_bits(unsigned x, unsigned bits) {
    unsigned r = 0;
    for (unsigned i = 0; i < bits; i++) r |= ((x >> i) & 1u) << (bits - 1 - i);
    return r;
}

// A matrix that exists as natural-order ROW blocks over the ranks (rows [d n / N, (d + 1) n / N) on rank d), or whole on every
// rank (block == the full matrix).
struct RowBlocks {
    size_t height = 0, width = 0;  // of the whole matrix
    bool whole = false;
    DevBuf own;                    // the buffer behind `dev`, empty when it is the caller's (msh_rowshard_commit)
    const uint64_t* dev = nullptr; // this rank's block (height / N rows) or the whole matrix
};

class RowShardOpenDevice;

class RowShardBackend : public ShardedBackend {
  public:
    RowShardBackend(msgpu_ctx* ctx, const SystemShape& shape, const msh_comm& comm) : ShardedBackend(ctx, shape, comm) {
        const int n = comm_.world();
        if (n < 1 || (n & (n - 1))) throw DistError("row-sharded prover: the number of ranks must be a power of two");
        if (n > 16) throw DistError("row-sharded prover: at most 16 ranks");
        // msgpu_stage2_trace evaluates the lookups of a row block as if the block were the whole trace: a next-row read would need
        // a one-row halo between the blocks, and the selectors would mark the block's first and last rows, not the trace's
        for (auto& c : shape_.circuits) {
            std::string& r = lookup_block_reads_.emplace_back();
            for (size_t i = 0; i < c.graph.lookup_prefix_len && r.empty(); i++) {
                const Node& nd = c.graph.nodes[i];
                if (nd.op == Op::Var && nd.col.offset == RowOffset::Next) r = "the next row";
                else if (nd.op == Op::IsFirstRow) r = "is_first_row";
                else if (nd.op == Op::IsLastRow) r = "is_last_row";
                else if (nd.op == Op::IsTransition) r = "is_transition";
            }
        }
        if (comm.peer_memory && n > 1) init_peers();
    }
    ~RowShardBackend() override {
        RowShardBackend::end_proof();
        if (peers_) msgpu_peers_destroy(peers_);
    }
    bool peer_memory() const { return peers_ != nullptr; }
    // bytes this rank wrote into / read from the other ranks' windows so far (matrix data; roots and flags not counted)
    uint64_t peer_bytes() const { return peer_bytes_; }
    // matrices that take the peer-memory path: split by columns for the NTT, and tall enough for a two-pass transform
    bool peer_path(size_t height, size_t width) const { return peers_ && shardable(height, width); }

    int world() const { return comm_.world(); }
    int rank() const { return comm_.rank(); }
    const CommView& comm() const { return comm_; }
    msgpu_ctx* ctx() const { return ctx_; }

    // wide and tall enough to be split by columns for the NTT and by rows afterwards
    // With peer memory any width is split (a rank may hold no column of a narrow matrix during the NTT: it still hashes its rows).
    bool shardable(size_t height, size_t width) const {
        if (world() <= 1) return false;
        if (peers_) return width >= 1 && height >= 2048 && height >= (size_t)world() * 64;
        return (int)width >= world() && height >= (size_t)world() * 64;
    }

    // ---- commitments ---------------------------------------------------------------------------------------------------
    // rows of this rank's shard of the LDE of `m` (shardable: column-sharded NTT between two all-to-alls; otherwise the whole LDE
    // on every rank). Returns the buffer to own; *view = this rank's rows.
    DevBuf lde_shard(const RowBlocks& m, uint64_t** view, bool* whole) {
        const int N = world(), d = rank();
        const uint32_t lb = (uint32_t)shape_.log_blowup();
        const size_t n = m.height, w = m.width, H = n << lb, Ls = H / (size_t)N;
        if (H < (size_t)N) throw DistError("row-sharded prover: a committed matrix has fewer LDE rows than there are ranks");
        if (!m.whole && !shardable(n, w)) throw DistError("row-sharded prover: internal error, row blocks of an unshardable matrix");
        if (m.whole) {
            DevBuf lde(ctx_, H * w * 8);
            if (w) gpu_check(msgpu_coset_lde_batch_bitrev_dev(ctx_, m.dev, n, w, lb, GL_GENERATOR, lde.get()));
            *view = lde.get() + (size_t)d * Ls * w;
            *whole = true;
            return lde;
        }
        // column blocks: the first w % N ranks get one more column
        std::vector<uint64_t> c0(N), c1(N), wd(N);
        {
            size_t base = w / N, rem = w % N, c = 0;
            for (int e = 0; e < N; e++) { c0[e] = c; c += base + ((size_t)e < rem ? 1 : 0); c1[e] = c; wd[e] = c1[e] - c0[e]; }
        }
        const size_t nb = n / (size_t)N;  // rows of a natural-order block
        DevBuf packed(ctx_, nb * w * 8), colblock(ctx_, n * wd[d] * 8);
        gpu_check(msgpu_pack_column_blocks_dev(ctx_, m.dev, nb, w, N, c0.data(), c1.data(), packed.get()));
        std::vector<uint64_t> sb(N), rb(N);
        for (int e = 0; e < N; e++) { sb[e] = nb * wd[e] * 8; rb[e] = nb * wd[d] * 8; }
        comm_.alltoall_dev(packed.get(), sb.data(), colblock.get(), rb.data());  // pieces arrive in rank order = natural row order
        packed.reset();
        DevBuf lde(ctx_, H * wd[d] * 8);
        gpu_check(msgpu_coset_lde_batch_bitrev_dev(ctx_, colblock.get(), n, wd[d], lb, GL_GENERATOR, lde.get()));
        colblock.reset();
        // rows [e Ls, (e + 1) Ls) of my columns are contiguous: chunk e goes to rank e
        DevBuf chunks(ctx_, Ls * w * 8);
        for (int e = 0; e < N; e++) { sb[e] = Ls * wd[d] * 8; rb[e] = Ls * wd[e] * 8; }
        comm_.alltoall_dev(lde.get(), sb.data(), chunks.get(), rb.data());
        lde.reset();
        DevBuf shard(ctx_, Ls * w * 8);
        gpu_check(msgpu_interleave_column_blocks_dev(ctx_, chunks.get(), Ls, N, wd.data(), shard.get()));
        *view = shard.get();
        *whole = false;
        return shard;
    }

    // MMCS over the shards: local subtree + replicated top
    std::shared_ptr<RowShardHandle> commit_shards(std::shared_ptr<RowShardHandle> h, Digest& root) {
        const int N = world();
        std::vector<uint64_t*> ptrs;
        std::vector<uint64_t> hs, ws;
        for (size_t i = 0; i < h->shapes.size(); i++) {
            if (h->shapes[i].first < (size_t)N) throw DistError("row-sharded prover: a committed matrix has fewer LDE rows than there are ranks");
            ptrs.push_back(h->views[i]);
            hs.push_back(h->shard_rows(i));
            ws.push_back(h->shapes[i].second);
        }
        msgpu_pdata* pd = nullptr;
        if (N == 1) {
            gpu_check(msgpu_commit_ldes_dev(ctx_, ptrs.data(), hs.data(), ws.data(), ptrs.size(), 0, &pd, root.data()));
            h->local.reset(pd);
            return h;
        }
        // views that are still column blocks in the peers' windows are assembled by the leaf-hash pass itself
        std::vector<const uint64_t*> bptr;
        std::vector<uint64_t> bwid;
        uint64_t n_blocks = 0;
        h->pending.resize(h->shapes.size());
        for (auto& pb : h->pending) n_blocks = std::max<uint64_t>(n_blocks, pb.size());
        if (n_blocks) {
            bptr.assign(ptrs.size() * n_blocks, nullptr);
            bwid.assign(ptrs.size() * n_blocks, 0);
            for (size_t i = 0; i < h->pending.size(); i++)
                for (size_t b = 0; b < h->pending[i].size(); b++) {
                    bptr[i * n_blocks + b] = h->pending[i][b].first;
                    bwid[i * n_blocks + b] = h->pending[i][b].second;
                }
        }
        // leaf digests + subtree, stream-ordered (no read-back); the 32-byte subtree roots are all-gathered on the device and the
        // top levels built from them: ONE host synchronisation per commitment, for the root the transcript needs
        gpu_check(msgpu_commit_ldes_blocks_dev(ctx_, ptrs.data(), hs.data(), ws.data(), ptrs.size(), n_blocks, n_blocks ? bptr.data() : nullptr,
                                               n_blocks ? bwid.data() : nullptr, 0, &pd, nullptr));
        h->local.reset(pd);
        h->pending.clear();
        uint8_t* dg = nullptr;
        uint64_t nd = 0;
        gpu_check(msgpu_pdata_digests(h->local.get(), &dg, &nd));
        uint64_t hh = (uint64_t)N;
        if (peers_) {
            // every rank stores its root into slot `rank` of every peer's ring entry; the flag barrier publishes them
            uint8_t* gathered = nullptr;
            gpu_check(msgpu_peers_put_root(peers_, dg + (nd - 1) * 32, &gathered));
            gpu_check(msgpu_peers_barrier(peers_));
            const uint8_t* pp = gathered;
            gpu_check(msgpu_tree_from_digests(ctx_, 1, &hh, &pp, &pd, root.data()));
            h->top.reset(pd);
            gpu_check(msgpu_peers_check(peers_));  // a barrier of this commitment timed out: fail here, not with a wrong root
            rs_trace(rank(), "root");
            return h;
        }
        DevBuf d_roots(ctx_, 32 * (size_t)N);
        comm_.allgather_dev(dg + (nd - 1) * 32, d_roots.get(), 32);
        const uint8_t* pp = (const uint8_t*)d_roots.get();
        gpu_check(msgpu_tree_from_digests(ctx_, 1, &hh, &pp, &pd, root.data()));
        h->top.reset(pd);
        return h;
    }

    std::shared_ptr<RowShardHandle> commit_blocks(const std::vector<RowBlocks>& mats, Digest& root) {
        auto h = std::make_shared<RowShardHandle>();
        h->n_shards = world();
        h->shard = rank();
        const uint32_t lb = (uint32_t)shape_.log_blowup();
        const size_t N = (size_t)world(), d = (size_t)rank();
        // Peer-memory matrices. Blocks of the symmetric heap, the same (segment, offset) on every rank: col = this rank's dense
        // column block of the evaluations (written by every rank), lde = its column block of the LDE (read by every rank).
        std::vector<SymBlock> col(mats.size()), lde(mats.size()), held;
        struct FreeHeld { RowShardBackend* b; std::vector<SymBlock>& v; ~FreeHeld() { for (auto& x : v) msgpu_peers_free_block(b->peers_, x.seg, x.off); } } fh{this, held};
        bool any_peer = false;
        rs_trace(rank(), "commit_blocks", mats.size());
        for (size_t i = 0; i < mats.size(); i++) {
            const RowBlocks& m = mats[i];
            if (m.whole || !peer_path(m.height, m.width)) continue;
            any_peer = true;
            const size_t wmax = (m.width + N - 1) / N;
            col[i] = sym_alloc(m.height * wmax * 8);
            held.push_back(col[i]);
            lde[i] = sym_alloc((m.height << lb) * wmax * 8);
            held.push_back(lde[i]);
            // my rows of every rank's column block: remote stores, contiguous per destination
            gpu_check(msgpu_peers_pack_push(peers_, m.dev, m.height / N, m.width, col[i].seg, col[i].off));
            {   // NVLink bytes of this matrix: rows pushed to the other ranks' column blocks + shard rows pulled from theirs
                const size_t w = m.width, base = w / N, rem = w % N, wd = base + (d < rem ? 1 : 0);
                peer_bytes_ += (m.height / N) * (w - wd) * 8 + ((m.height << lb) / N) * (w - wd) * 8;
            }
        }
        rs_trace(rank(), "pushed");
        if (any_peer) gpu_check(msgpu_peers_barrier(peers_));  // every rank's rows have landed in this rank's column blocks
        for (size_t i = 0; i < mats.size(); i++) {
            const RowBlocks& m = mats[i];
            if (!col[i].live) continue;
            const size_t w = m.width, base = w / N, rem = w % N, wd = base + (d < rem ? 1 : 0);
            if (wd == 0) continue;  // a matrix narrower than the number of ranks: this rank extends no column of it
            gpu_check(msgpu_coset_lde_batch_bitrev_dev(ctx_, sym_ptr(col[i]), m.height, wd, lb, GL_GENERATOR, sym_ptr(lde[i])));
        }
        if (any_peer) gpu_check(msgpu_peers_barrier(peers_));  // every rank's column block of every LDE is complete
        for (size_t i = 0; i < mats.size(); i++) {
            const RowBlocks& m = mats[i];
            uint64_t* view = nullptr;
            bool whole = false;
            if (col[i].live) {
                // my row shard from every rank's column block: remote loads of whole lines
                const size_t Ls = (m.height << lb) / N;
                h->owned.emplace_back(ctx_, Ls * m.width * 8);
                view = h->owned.back().get();
                // ... inside the pass that hashes them (commit_shards): block e = rank e's columns of my rows
                std::vector<std::pair<const uint64_t*, uint64_t>> blocks;
                const size_t base = m.width / N, rem = m.width % N;
                for (size_t e = 0; e < N; e++) {
                    const size_t wde = base + (e < rem ? 1 : 0);
                    const uint64_t* p = (const uint64_t*)msgpu_peers_ptr(peers_, lde[i].seg, lde[i].off, (int32_t)e);
                    if (!p) throw DistError("peer heap: internal error, unmapped block");
                    blocks.push_back({p + d * Ls * wde, wde});
                }
                h->pending.resize(i + 1);
                h->pending[i] = std::move(blocks);
            } else {
                h->owned.push_back(lde_shard(m, &view, &whole));
            }
            h->views.push_back(view);
            h->whole.push_back(whole);
            h->shapes.push_back({m.height << lb, m.width});
        }
        rs_trace(rank(), "ldes done");
        // the root barrier inside commit_shards orders every rank's loads from the column blocks before their release
        return commit_shards(h, root);
    }

    // upload of a host matrix every rank can read: its natural-order row block when shardable, all of it otherwise
    RowBlocks upload_blocks(const uint64_t* host, size_t height, size_t width) {
        RowBlocks b;
        b.height = height;
        b.width = width;
        b.whole = !shardable(height, width);
        const size_t rows = b.whole ? height : height / (size_t)world(), row0 = b.whole ? 0 : rows * (size_t)rank();
        b.own = upload(host + row0 * width, rows * width);
        b.dev = b.own.get();
        return b;
    }

    // System::new: the preprocessed commitment (src/system.rs:180-196)
    PcsHandlePtr commit(const std::vector<const Matrix*>& evals, Digest& root) override {
        std::vector<RowBlocks> mats;
        for (auto* m : evals) mats.push_back(upload_blocks((const uint64_t*)m->values.data(), m->height(), m->width));
        return commit_blocks(mats, root);
    }

    PcsHandlePtr commit_stage1(const std::vector<size_t>& circuits, const std::vector<MatrixView>& traces, Digest& root) override {
        end_proof();
        active_ = circuits;
        claims_rank_ = world() - 1;  // not the FRI owner
        if (rank() != claims_rank_) announced_ = ClaimsView();
        for (size_t p = 0; p < circuits.size(); p++) {
            const MatrixView& m = traces[p];
            if (!m.data) throw DistError("row-sharded prover: every rank needs (read access to) every trace");
            trace_rows_.push_back(m.height());
            const std::string& reads = lookup_block_reads_[circuits[p]];
            if (!reads.empty() && shardable(m.height(), m.width))
                throw DistError("row-sharded prover: lookups that read " + reads + " are not supported on row blocks");
            main_.push_back(upload_blocks((const uint64_t*)m.data, m.height(), m.width));
        }
        prefetch_announced_claims();
        return commit_blocks(main_, root);
    }

    PcsHandlePtr commit_stage2(Fp2 beta, Fp2 gamma, Fp2 acc, std::vector<Fp2>& intermediate, Digest& root) override {
        const int N = world(), d = rank();
        uint64_t b[2] = {beta.c[0].v, beta.c[1].v}, g[2] = {gamma.c[0].v, gamma.c[1].v};
        std::vector<RowBlocks> s2;
        std::vector<uint64_t> sums(2 * active_.size(), 0);
        for (size_t p = 0; p < active_.size(); p++) {
            const Circuit& c = shape_.circuits[active_[p]];
            const RowBlocks& mt = main_[p];
            const size_t rows = mt.whole ? mt.height : mt.height / (size_t)N, row0 = mt.whole ? 0 : rows * (size_t)d;
            RowBlocks out;
            out.height = mt.height;
            out.width = c.stage_2_width;
            out.whole = mt.whole;
            out.own = DevBuf(ctx_, rows * c.stage_2_width * 8);
            out.dev = out.own.get();
            uint64_t* dst = out.own.get();
            s2.push_back(std::move(out));
            const uint64_t* pre = pre_dev_[active_[p]].get() ? pre_dev_[active_[p]].get() + row0 * c.preprocessed_width : nullptr;
            gpu_check(msgpu_stage2_trace(ctx_, programs_[active_[p]], pre, mt.dev, rows, b, g, dst, &sums[2 * p]));
        }
        // the ranks' totals: offsets of the row blocks' running sums, and the circuits' totals for the accumulator chain
        std::vector<uint64_t> all(sums.size() * (size_t)N);
        rs_trace(d, "stage2 sums allgather");
        comm_.allgather(sums.data(), all.data(), sums.size() * 8);
        intermediate.clear();
        for (size_t p = 0; p < active_.size(); p++) {
            const Circuit& c = shape_.circuits[active_[p]];
            Fp2 total, offset;
            if (s2[p].whole) {
                total = Fp2(Fp(all[2 * p]), Fp(all[2 * p + 1]));  // every rank computed the whole trace: rank 0's total
            } else {
                for (int e = 0; e < N; e++) {
                    Fp2 t(Fp(all[(size_t)e * sums.size() + 2 * p]), Fp(all[(size_t)e * sums.size() + 2 * p + 1]));
                    if (e < d) offset += t;
                    total += t;
                }
                if (!offset.is_zero()) {
                    uint64_t o2[2] = {offset.c[0].v, offset.c[1].v};
                    gpu_check(msgpu_ext_add_scalar_dev(ctx_, s2[p].own.get(), (s2[p].height / (size_t)N) * (c.stage_2_width / 2), o2));
                }
            }
            acc += total;
            intermediate.push_back(acc);
        }
        // a block-built stage-2 trace that is too narrow to be split by columns is made whole on every rank
        for (size_t p = 0; p < s2.size(); p++) {
            if (s2[p].whole || shardable(s2[p].height, s2[p].width)) continue;
            const size_t nb = s2[p].height / (size_t)N, w = s2[p].width;
            DevBuf full(ctx_, s2[p].height * w * 8);
            comm_.allgather_dev(s2[p].own.get(), full.get(), nb * w * 8);
            s2[p].own = std::move(full);
            s2[p].dev = s2[p].own.get();
            s2[p].whole = true;
        }
        auto h = commit_blocks(s2, root);
        main_.clear();
        return h;
    }

    PcsHandlePtr commit_quotient(const std::vector<QuotientJob>& jobs, PcsHandle* pre, PcsHandle* s1, PcsHandle* s2, Fp2 alpha,
                                 Digest& root) override {
        auto* h1 = dynamic_cast<RowShardHandle*>(s1);
        auto* h2 = dynamic_cast<RowShardHandle*>(s2);
        auto* hp = pre ? dynamic_cast<RowShardHandle*>(pre) : nullptr;
        if (!h1 || !h2 || (pre && !hp)) throw DistError("quotient: prover data does not belong to the row-sharded backend");
        const int N = world(), d = rank();
        const uint32_t lb = (uint32_t)shape_.log_blowup();
        uint64_t a[2] = {alpha.c[0].v, alpha.c[1].v};
        auto h = std::make_shared<RowShardHandle>();
        h->n_shards = N;
        h->shard = d;
        for (auto& j : jobs) {
            rs_trace(rank(), "quotient job", j.circuit, j.log_degree);
            const size_t H = (size_t)1 << (j.log_degree + lb), Ls = H / (size_t)N, nq = (size_t)1 << (j.log_degree + j.log_quotient_degree);
            const size_t q = (size_t)1 << j.log_quotient_degree;
            // shards spanning the quotient domain, the rows of it held here, and the shard that holds their next rows
            const size_t Np = std::max<size_t>(1, nq / Ls);
            const unsigned lnp = log2_strict(Np);
            const size_t row0 = (size_t)d * Ls, n_local = row0 >= nq ? 0 : std::min(Ls, nq - row0);
            auto next_of = [&](size_t e) { return (size_t)rs_rev_bits((unsigned)((rs_rev_bits((unsigned)e, lnp) + q) & (Np - 1)), lnp); };
            struct Src { RowShardHandle* h; size_t idx; };
            Src src[3] = {{hp, j.preprocessed_idx >= 0 ? (size_t)j.preprocessed_idx : 0}, {h1, j.pos}, {h2, j.pos}};
            const bool has_pre = j.preprocessed_idx >= 0 && hp;
            const uint64_t* cur[3] = {nullptr, nullptr, nullptr};
            const uint64_t* nxt[3] = {nullptr, nullptr, nullptr};
            uint32_t nw[3] = {0, 0, 0}, nc0[3] = {0, 0, 0};
            // the columns each source is read at with the NEXT-row offset: the stage-2 accumulator pair (the logUp wrap /
            // pass-through constraint reads stage2_next[0..2], src/lookup.rs:167-208) and whatever the constraints name
            size_t lo[3] = {SIZE_MAX, SIZE_MAX, 0}, hi[3] = {0, 0, 2};
            for (auto& nd : shape_.circuits[j.circuit].graph.nodes)
                if (nd.op == Op::Var && nd.col.offset == RowOffset::Next) {
                    const int k = (int)nd.col.source;
                    lo[k] = std::min<size_t>(lo[k], nd.col.index);
                    hi[k] = std::max<size_t>(hi[k], (size_t)nd.col.index + 1);
                }
            std::vector<DevBuf> halos;
            size_t next_row0 = row0;
            const size_t dn = (size_t)d < Np ? next_of((size_t)d) : (size_t)d;
            if ((size_t)d < Np) next_row0 = dn * Ls;
            for (int k = 0; k < 3; k++) {
                if (k == 0 && !has_pre) continue;
                RowShardHandle* sh = src[k].h;
                const size_t i = src[k].idx, w = sh->shapes[i].second;
                if (sh->shapes[i].first != H) throw DistError("quotient: the circuit's committed matrices differ in height");
                cur[k] = sh->views[i];
                nxt[k] = sh->views[i];  // never read when the source has no next-row reference
                nw[k] = (uint32_t)w;
                // every condition that skips the exchange must hold on ALL ranks alike (a collective under NCCL): no next-row
                // reference, the whole matrix here, or a trace step that stays inside the shard (q = 0 mod Np)
                if (lo[k] >= hi[k]) continue;
                if (sh->whole[i]) {
                    if (dn != (size_t)d) nxt[k] = sh->whole_rows_of(i, (int)dn);
                    continue;
                }
                if (Np > 1 && (q & (Np - 1)) != 0) {
                    // fetch columns [lo, hi) of shard dn: rank e sends those columns of its quotient-domain rows to the rank whose
                    // next rows they are (a permutation of the ranks: one all-to-all call)
                    const size_t wc = hi[k] - lo[k], rows = std::min(Ls, nq), bytes = rows * wc * 8;
                    std::vector<uint64_t> sb(N, 0), rb(N, 0);
                    DevBuf packed(ctx_, bytes);
                    bool need = false;
                    if ((size_t)d < Np && dn != (size_t)d) {
                        for (size_t e = 0; e < Np; e++)
                            if (next_of(e) == (size_t)d && e != (size_t)d) sb[e] = bytes;
                        gpu_check(msgpu_extract_columns_dev(ctx_, sh->views[i], rows, w, lo[k], hi[k], packed.get()));
                        rb[dn] = bytes;
                        need = true;
                    }
                    halos.emplace_back(ctx_, need ? bytes : 8);
                    rs_trace(rank(), "halo a2a", (size_t)k, bytes);
                    comm_.alltoall_dev(packed.get(), sb.data(), halos.back().get(), rb.data());
                    if (need) {
                        nxt[k] = halos.back().get();
                        nw[k] = (uint32_t)wc;
                        nc0[k] = (uint32_t)lo[k];
                    }
                }
            }
            // quotient evaluations of the local rows (stored order) -> all ranks -> the 2q-column quotient LDE on every rank
            DevBuf mine(ctx_, std::max<size_t>(Ls * 16, 16)), all(ctx_, (size_t)N * Ls * 16);
            uint64_t pub[8];
            for (int k = 0; k < 8; k++) pub[k] = j.publics[k].v;
            gpu_check(msgpu_quotient_values_shard(ctx_, programs_[j.circuit], cur, nxt, nw, nc0, row0, n_local, next_row0, j.log_degree,
                                                  j.log_quotient_degree, pub, a, mine.get()));
            halos.clear();
            rs_trace(rank(), "quotient values allgather", Ls * 16);
            comm_.allgather_dev(mine.get(), all.get(), Ls * 16);  // the first nq rows of the result are the quotient domain
            uint64_t* lde = nullptr;
            gpu_check(msgpu_quotient_finish(ctx_, all.get(), j.log_degree, j.log_quotient_degree, lb, &lde));
            h->owned.emplace_back(ctx_, lde);
            h->views.push_back(lde + (size_t)d * Ls * (2 * q));
            h->whole.push_back(true);
            h->shapes.push_back({H, 2 * q});
        }
        return commit_shards(h, root);
    }

    std::unique_ptr<OpenDevice> open_begin(const std::vector<OpenRound>& rounds) override;

    void end_proof() override {
        GpuBackend::end_proof();
        main_.clear();
    }

    // ---- the symmetric peer heap -----------------------------------------------------------------------------------------
    // Every rank makes the same calls with the same sizes, so the deterministic allocator returns the same (segment, offset)
    // everywhere. A request that fits nowhere grows the heap by one window on all ranks at once (handles all-gathered on the host).
    SymBlock sym_alloc(size_t bytes) {
        SymBlock b;
        int rc = msgpu_peers_alloc(peers_, bytes, &b.seg, &b.off);
        if (rc == 1) {
            sym_grow(bytes);
            rc = msgpu_peers_alloc(peers_, bytes, &b.seg, &b.off);
            if (rc == 1) throw DistError("peer heap: internal error, a fresh window cannot hold the block it was made for");
        }
        gpu_check(rc);
        b.live = true;
        return b;
    }
    uint64_t* sym_ptr(const SymBlock& b) const { return (uint64_t*)msgpu_peers_ptr(peers_, b.seg, b.off, comm_.rank()); }

  private:
    // collective; returns false when any rank failed (the heap is then unusable on every rank)
    bool sym_grow_try(size_t need) {
        const int N = world();
        size_t bytes = std::max<size_t>(need + (1u << 16), (size_t)1 << 30);
        if (const char* e = getenv("MSGPU_PEER_WINDOW_MB")) bytes = std::max<size_t>(need + (1u << 16), (size_t)atoll(e) << 20);
        bytes = (bytes + ((size_t)1 << 21) - 1) >> 21 << 21;
        std::vector<uint8_t> mine(72, 0), all(72 * (size_t)N);
        int32_t rc = msgpu_peers_segment_create(peers_, bytes, mine.data());
        memcpy(mine.data() + 64, &rc, 4);
        comm_.allgather(mine.data(), all.data(), 72);
        std::vector<uint8_t> handles(64 * (size_t)N);
        bool ok = true;
        for (int e = 0; e < N; e++) {
            int32_t r;
            memcpy(&r, all.data() + 72 * (size_t)e + 64, 4);
            ok = ok && r == 0;
            memcpy(handles.data() + 64 * (size_t)e, all.data() + 72 * (size_t)e, 64);
        }
        int32_t rc2 = ok ? msgpu_peers_segment_open(peers_, handles.data()) : -1;
        std::vector<int32_t> rcs(N);
        comm_.allgather(&rc2, rcs.data(), 4);
        for (int32_t r : rcs) ok = ok && r == 0;
        return ok;
    }
    void sym_grow(size_t need) {
        if (!sym_grow_try(need)) throw DistError(std::string("peer heap: a window could not be created or mapped on every rank: ") + msgpu_last_error());
    }
    void init_peers() {
        gpu_check(msgpu_peers_create(ctx_, comm_.rank(), comm_.world(), &peers_));
        if (!sym_grow_try(0)) {  // no CUDA IPC between these processes: every rank falls back to the collectives
            msgpu_peers_destroy(peers_);
            peers_ = nullptr;
            if (getenv("MSH_TRACE")) fprintf(stderr, "[rowshard] rank %d: peer memory unavailable (%s), using collectives\n", comm_.rank(), msgpu_last_error());
        }
    }
    msgpu_peers* peers_ = nullptr;
    uint64_t peer_bytes_ = 0;
    std::vector<RowBlocks> main_;  // the natural-order traces (row blocks or whole), kept for the stage-2 construction
    std::vector<std::string> lookup_block_reads_;  // per circuit: what its lookups read that a row block cannot evaluate ("" = nothing)
};

// Pcs::open over the row shards.
class RowShardOpenDevice : public ShardedOpenDevice {
  public:
    RowShardOpenDevice(RowShardBackend& be, const std::vector<OpenRound>& rounds, uint32_t log_blowup) : ShardedOpenDevice(be.ctx(), be.comm(), rounds) {
        const int N = comm_.world(), d = comm_.rank();
        std::vector<const msgpu_pdata*> pds;
        std::vector<uint32_t> modes;
        std::vector<uint64_t> npts, pts;
        size_t max_h = 0;
        for (auto& r : rounds) {
            auto* h = dynamic_cast<RowShardHandle*>(r.data);
            if (!h) throw DistError("open: prover data does not belong to the row-sharded backend");
            if (r.points.size() != h->shapes.size()) throw DistError("open: one point list per committed matrix expected");
            handles_.push_back(h);
            pds.push_back(h->local.get());
            modes.push_back(1);
            for (size_t m = 0; m < h->shapes.size(); m++) {
                max_h = std::max(max_h, h->shapes[m].first);
                npts.push_back(r.points[m].size());
                for (auto& z : r.points[m]) { pts.push_back(z.c[0].v); pts.push_back(z.c[1].v); }
            }
        }
        log_max_height_ = log2_strict(max_h);
        if (pts.empty()) pts.push_back(0);
        uint64_t n_sums = 0;
        gpu_check(msgpu_open_begin_shard(ctx_, pds.size(), pds.data(), modes.data(), (uint32_t)d, (uint32_t)N, d == fri_owner_ ? 1 : 0, npts.data(),
                                         pts.data(), log_blowup, &op_, &n_values_, &n_sums));
        rs_trace(d, "open_begin done", n_sums);
        // barycentric sums of all ranks, added in the field
        std::vector<uint64_t> mine(std::max<uint64_t>(n_sums, 1)), all((size_t)N * std::max<uint64_t>(n_sums, 1));
        gpu_check(msgpu_open_sums(op_, mine.data()));
        comm_.allgather(mine.data(), all.data(), mine.size() * 8);
        for (uint64_t i = 0; i < n_sums; i++) {
            Fp s;
            for (int e = 0; e < N; e++) s += Fp(all[(size_t)e * mine.size() + i]);
            mine[i] = s.v;
        }
        gpu_check(msgpu_open_finish_values(op_, mine.data()));
    }

    std::vector<OpenedValuesForRound> evaluate() override {
        std::vector<uint64_t> flat(std::max<size_t>(2 * n_values_, 1));
        gpu_check(msgpu_open_values(op_, flat.data()));
        return decode_opened_values(rounds_, flat.data());
    }

    void reduce(Fp2 alpha, unsigned& log_max_height) override {
        const int N = comm_.world(), d = comm_.rank();
        uint64_t a[2] = {alpha.c[0].v, alpha.c[1].v}, n_in = 0;
        uint32_t lm = 0;
        rs_trace(d, "reduce");
        gpu_check(msgpu_open_reduce(op_, a, &n_in, &lm));
        // every rank holds rows of every height: the shards (16 bytes per LDE row) are added into the owner's full-length vectors
        for (uint64_t k = 0; k < n_in && N > 1; k++) {
            uint64_t* p = nullptr;
            uint64_t len = 0;
            gpu_check(msgpu_open_input_dev(op_, k, &p, &len));
            const uint64_t Ls = d == fri_owner_ ? len / (uint64_t)N : len;
            std::vector<uint64_t> sb(N, 0), rb(N, 0);
            if (d == fri_owner_) {
                for (int e = 0; e < N; e++)
                    if (e != fri_owner_) rb[e] = Ls * 16;
                DevBuf tmp(ctx_, (uint64_t)(N - 1) * Ls * 16);
                comm_.alltoall_dev(p, sb.data(), tmp.get(), rb.data());
                // chunks arrive in rank order; the owner is rank 0, so they are the rows from Ls on
                gpu_check(msgpu_ext_add_dev(ctx_, p + 2 * Ls, tmp.get(), (uint64_t)(N - 1) * Ls));
                gpu_check(msgpu_sync(ctx_));
            } else {
                sb[fri_owner_] = Ls * 16;
                comm_.alltoall_dev(p, sb.data(), p, rb.data());  // nothing is received
            }
        }
        cur_len_ = size_t(1) << log_max_height_;
        log_max_height = log_max_height_;
    }
  protected:
    // the device transcript when there is no proof of work, otherwise the host loop
    void owner_commit_phase(Challenger& ch, size_t stop_len, size_t pow_bits, FriProof& proof) override {
        if (!fri_commit_phase_on_device(op_, cur_len_, ch, stop_len, pow_bits, proof, betas)) OpenDevice::commit_phase(ch, stop_len, pow_bits, proof);
    }

  public:
    // Rows and the lower log2(H / N) siblings of a query come from the rank that holds the row, the top log2 N siblings from the
    // top tree (on every rank); the FRI layers from the owner. One all-gather of every rank's share.
    void open_queries(const std::vector<size_t>& indices, const std::vector<unsigned>& round_shifts, size_t n_layers,
                      std::vector<std::vector<BatchOpening>>& rounds_out, std::vector<std::vector<BatchOpening>>& layers_out) override {
        const int N = comm_.world(), d = comm_.rank();
        const size_t n = indices.size(), R = handles_.size();
        rs_trace(d, "open_queries", n, R);
        const unsigned log_n_shards = log2_strict((size_t)N);
        // per round: the round's index of every query, its holder and the index inside the holder's shard
        std::vector<std::vector<size_t>> ridx(R, std::vector<size_t>(n)), holder(R, std::vector<size_t>(n));
        std::vector<size_t> Ls(R), tw(R, 0), lo_depth(R);
        for (size_t r = 0; r < R; r++) {
            Ls[r] = ((size_t(1) << log_max_height_) >> round_shifts[r]) / (size_t)N;
            lo_depth[r] = log2_strict(Ls[r]);
            for (auto& s : handles_[r]->shapes) tw[r] += s.second;
            for (size_t q = 0; q < n; q++) {
                ridx[r][q] = indices[q] >> round_shifts[r];
                holder[r][q] = ridx[r][q] / Ls[r];
            }
        }
        // my share: for every round the queries I hold (rows of all its matrices + lower path), then the layers if I am the owner
        std::vector<u8> blob;
        for (size_t r = 0; r < R; r++) {
            std::vector<uint64_t> mine;
            for (size_t q = 0; q < n; q++)
                if (holder[r][q] == (size_t)d) mine.push_back(ridx[r][q] % Ls[r]);
            if (mine.empty()) continue;
            std::vector<uint64_t> opened(mine.size() * std::max<size_t>(tw[r], 1));
            std::vector<uint8_t> paths(std::max<size_t>(mine.size() * lo_depth[r] * 32, 1));
            gpu_check(msgpu_open_batch(ctx_, handles_[r]->local.get(), mine.data(), mine.size(), opened.data(), paths.data()));
            const size_t ob = mine.size() * tw[r] * 8, pb = mine.size() * lo_depth[r] * 32;
            const size_t at = blob.size();
            blob.resize(at + ob + pb);
            if (ob) memcpy(blob.data() + at, opened.data(), ob);
            if (pb) memcpy(blob.data() + at + ob, paths.data(), pb);
        }
        // every rank can compute every rank's share size (the holders follow from the indices): ONE all-gather, padded to the largest
        std::vector<size_t> share(N, 0);
        for (size_t r = 0; r < R; r++)
            for (size_t q = 0; q < n; q++) share[holder[r][q]] += tw[r] * 8 + lo_depth[r] * 32;
        if (share[d] != blob.size()) throw DistError("open: internal error, query share size");
        size_t mx = 8;
        for (size_t sz : share) mx = std::max(mx, sz);
        std::vector<u8> sendbuf(mx, 0), recvbuf(mx * (size_t)N);
        if (!blob.empty()) memcpy(sendbuf.data(), blob.data(), blob.size());
        comm_.allgather(sendbuf.data(), recvbuf.data(), mx);
        std::vector<std::vector<u8>> all(N);
        for (int e = 0; e < N; e++) all[e].assign(recvbuf.begin() + (size_t)e * mx, recvbuf.begin() + (size_t)e * mx + share[e]);
        // the commit-phase layers live on the FRI owner: one broadcast of their openings
        layers_out.clear();
        if (n_layers) {
            std::vector<const msgpu_pdata*> trees;
            std::vector<uint32_t> shifts;
            std::vector<TreeShape> shapes;
            for (size_t k = 0; k < n_layers; k++) {
                if (d == fri_owner_) {
                    trees.push_back(fri_layer(op_, k));
                    shifts.push_back((uint32_t)(k + 1));
                }
                shapes.push_back(TreeShape{{4}, (size_t)(log_max_height_ - k - 1)});
            }
            std::vector<u8> layer_blob = d == fri_owner_ ? open_batch_multi(ctx_, trees, shifts, shapes, indices) : std::vector<u8>(batch_bytes(shapes, n));
            comm_.bcast(layer_blob.data(), layer_blob.size(), fri_owner_);
            layers_out = decode_batch_openings(shapes, n, layer_blob);
        }
        // the top siblings of every (round, query): the top tree's leaf is the holder's subtree root
        std::vector<std::vector<uint8_t>> top_paths(R);
        for (size_t r = 0; r < R && N > 1; r++) {
            std::vector<uint64_t> tidx(holder[r].begin(), holder[r].end());
            top_paths[r].resize(n * log_n_shards * 32);
            uint64_t dummy = 0;
            gpu_check(msgpu_open_batch(ctx_, handles_[r]->top.get(), tidx.data(), n, &dummy, top_paths[r].data()));
        }
        rounds_out.assign(R, std::vector<BatchOpening>(n));
        std::vector<size_t> cursor(N, 0);
        for (size_t r = 0; r < R; r++) {
            // the holders' shares list their queries in query order: walk them with one cursor per rank
            std::vector<size_t> cnt(N, 0), seen(N, 0);
            for (size_t q = 0; q < n; q++) cnt[holder[r][q]]++;
            for (size_t q = 0; q < n; q++) {
                const size_t e = holder[r][q];
                const u8* base = all[e].data() + cursor[e];
                const u8* rowp = base + seen[e] * tw[r] * 8;
                const u8* pathp = base + cnt[e] * tw[r] * 8 + seen[e] * lo_depth[r] * 32;
                if (cursor[e] + cnt[e] * (tw[r] * 8 + lo_depth[r] * 32) > all[e].size()) throw DistError("open: a rank sent a query share of unexpected size");
                BatchOpening& bo = rounds_out[r][q];
                for (auto& s : handles_[r]->shapes) {
                    std::vector<Fp> row(s.second);
                    if (s.second) memcpy(row.data(), rowp, s.second * 8);
                    rowp += s.second * 8;
                    bo.opened_values.push_back(std::move(row));
                }
                bo.opening_proof.resize(lo_depth[r] + (N > 1 ? log_n_shards : 0));
                for (size_t l = 0; l < lo_depth[r]; l++) memcpy(bo.opening_proof[l].data(), pathp + 32 * l, 32);
                for (size_t l = 0; N > 1 && l < log_n_shards; l++)
                    memcpy(bo.opening_proof[lo_depth[r] + l].data(), top_paths[r].data() + (q * log_n_shards + l) * 32, 32);
                seen[e]++;
            }
            for (int e = 0; e < N; e++) cursor[e] += cnt[e] * (tw[r] * 8 + lo_depth[r] * 32);
        }
    }

  private:
    uint64_t n_values_ = 0;
    std::vector<RowShardHandle*> handles_;
};

inline std::unique_ptr<OpenDevice> RowShardBackend::open_begin(const std::vector<OpenRound>& rounds) {
    return std::make_unique<RowShardOpenDevice>(*this, rounds, (uint32_t)shape_.log_blowup());
}

}  // namespace msh
