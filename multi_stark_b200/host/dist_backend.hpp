// One proof over several GPUs (SURVEY 8e, partitioning A: circuits -> ranks; BASELINE configs[3]).
//
// One process per GPU; every rank runs the SAME prove() driver (prover.hpp) with a replicated Fiat-Shamir transcript, over
// this backend, which does the heavy stages for the circuits it owns and exchanges only what the protocol forces:
//   * Pcs::commit (stage 1, stage 2, quotient, preprocessed): each rank builds the LDEs of its circuits and hashes the leaf
//     digests of its height classes; the 32-byte-per-row class digests go to the rank that owns the tallest class, which
//     builds the node layers (injection of the shorter classes, p3-merkle-tree) and broadcasts the root;
//   * logUp: every rank sums its circuits' terms; the per-circuit sums (16 B each) are all-gathered and chained into the
//     intermediate accumulators (src/prover.rs:391-409, src/lookup.rs:530-543);
//   * Pcs::open: opened values are all-gathered (a few KB); after alpha each rank reduces its own height classes (p3-fri keeps
//     one alpha-power counter per height, so a class that lives on one rank is reduced there exactly as on one GPU); the
//     reduced vectors (16 B per LDE row) go to the FRI owner, which runs the fold-and-commit rounds alone and broadcasts the
//     roots, PoW witnesses and the folded vector ONCE (the other ranks replay the transcript); query rows come from the
//     matrices' owners, sibling paths from the tree owners, and are all-gathered.
// Rule: all circuits of one trace height live on one rank (their rows share leaf digests and reduced openings).
// The proof is byte-identical to the single-GPU proof (tests/test_gpu_dist_prove.py).
#pragma once
#include "gpu_backend.hpp"
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <set>

extern "C" {
// Collectives supplied by the caller (Python: torch.distributed over NCCL / gloo, multi_stark_b200/dist.py). Every function
// returns 0 on success. Device buffers are valid in stream order of the context's stream; a call returns once the buffer may
// be used by work enqueued on that stream afterwards.
typedef struct msh_comm {
    void* user;
    int32_t rank, world;
    int (*allgather_host)(void* user, const void* send, void* recv, uint64_t bytes_per_rank);
    int (*bcast_host)(void* user, void* buf, uint64_t bytes, int32_t root);
    // called on `src` (sends) and on `dst` (receives) only
    int (*sendrecv_dev)(void* user, void* dev, uint64_t bytes, int32_t src, int32_t dst);
    // Device collectives of the row-sharded prover (rowshard_backend.hpp; may be NULL for the circuit-sharded one), called on
    // every rank. all-to-all: chunk e of `send` (send_bytes[e] bytes, chunks back to back in rank order) goes to rank e, chunk e
    // of `recv` comes from rank e. all-gather: `recv` receives world chunks of `bytes` in rank order.
    int (*alltoall_dev)(void* user, void* send, const uint64_t* send_bytes, void* recv, const uint64_t* recv_bytes);
    int (*allgather_dev)(void* user, void* send, void* recv, uint64_t bytes);
    // 1 = every rank drives its own GPU of ONE node and the processes may map each other's device memory (CUDA IPC): the
    // row-sharded prover then moves its matrices with NVLink loads / stores from inside its kernels (csrc/peer.cu) and keeps the
    // callbacks above for the small host-side exchanges. 0 = collectives only (gloo tests, several ranks on one device).
    int32_t peer_memory;
} msh_comm;
}

namespace msh {

struct DistError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

struct CommView {
    msh_comm c;
    int rank() const { return c.rank; }
    int world() const { return c.world; }
    void allgather(const void* send, void* recv, size_t bytes) const {
        if (c.allgather_host(c.user, send, recv, bytes) != 0) throw DistError("comm: allgather failed");
    }
    void bcast(void* buf, size_t bytes, int root) const {
        if (bytes && c.bcast_host(c.user, buf, bytes, root) != 0) throw DistError("comm: broadcast failed");
    }
    void sendrecv_dev(void* dev, size_t bytes, int src, int dst) const {
        if (c.sendrecv_dev(c.user, dev, bytes, src, dst) != 0) throw DistError("comm: device send/recv failed");
    }
    void alltoall_dev(void* send, const uint64_t* send_bytes, void* recv, const uint64_t* recv_bytes) const {
        if (!c.alltoall_dev) throw DistError("comm: the communicator has no device all-to-all");
        if (c.alltoall_dev(c.user, send, send_bytes, recv, recv_bytes) != 0) throw DistError("comm: device all-to-all failed");
    }
    // recv holds world() chunks of `bytes` in rank order; chunk rank() is `send`
    void allgather_dev(void* send, void* recv, uint64_t bytes) const {
        if (!c.allgather_dev) throw DistError("comm: the communicator has no device all-gather");
        if (bytes && c.allgather_dev(c.user, send, recv, bytes) != 0) throw DistError("comm: device all-gather failed");
    }
    // all-gather of byte strings of different lengths
    std::vector<std::vector<u8>> allgather_var(const std::vector<u8>& mine) const {
        std::vector<uint64_t> sizes(world());
        uint64_t n = mine.size();
        allgather(&n, sizes.data(), 8);
        size_t mx = 8;
        for (auto s : sizes) mx = std::max<size_t>(mx, s);
        std::vector<u8> send(mx, 0), recv(mx * world());
        if (n) memcpy(send.data(), mine.data(), n);
        allgather(send.data(), recv.data(), mx);
        std::vector<std::vector<u8>> out(world());
        for (int r = 0; r < world(); r++) out[r].assign(recv.begin() + (size_t)r * mx, recv.begin() + (size_t)r * mx + sizes[r]);
        return out;
    }
};

// MSH_TRACE=2: one line per protocol step and rank on stderr (a rank that stops printing is where a multi-GPU run hangs)
inline void rs_trace(int rank, const char* what, size_t a = 0, size_t b = 0) {
    static const bool on = getenv("MSH_TRACE") && atoi(getenv("MSH_TRACE")) >= 2;
    if (on) {
        fprintf(stderr, "[rs %d] %s %zu %zu\n", rank, what, a, b);
        fflush(stderr);
    }
}

// What the circuit-sharded and the row-sharded backends share: the communicator, and the claims (global, not sharded), which
// ONE rank uploads, hashes and accumulates -- the others receive 32 + 16 bytes. Each backend picks claims_rank_ in commit_stage1.
class ShardedBackend : public GpuBackend {
  public:
    bool observe_claims(Challenger& ch, const ClaimsView& claims) override {
        if (!claims_on_device(claims)) return GpuBackend::observe_claims(ch, claims);  // small set: every rank runs the host loop
        Digest d{};
        if (comm_.rank() == claims_rank_ && !claims_transcript_digest(ch.input_buffer(), claims, d))
            throw DistError("claims: internal error, device path refused");
        comm_.bcast(d.data(), 32, claims_rank_);
        ch.set_flushed(d);
        return true;
    }
    Fp2 claims_accumulator(const ClaimsView& claims, Fp2 beta, Fp2 gamma) override {
        if (!claims_on_device(claims)) return GpuBackend::claims_accumulator(claims, beta, gamma);
        uint64_t out[2] = {0, 0};
        if (comm_.rank() == claims_rank_) {
            Fp2 a = GpuBackend::claims_accumulator(claims, beta, gamma);
            out[0] = a.c[0].v;
            out[1] = a.c[1].v;
        }
        comm_.bcast(out, 16, claims_rank_);
        return Fp2(Fp(out[0]), Fp(out[1]));
    }

  protected:
    ShardedBackend(msgpu_ctx* ctx, const SystemShape& shape, const msh_comm& comm) : GpuBackend(ctx, shape), comm_{comm} {}
    CommView comm_;
    int claims_rank_ = 0;
};

// What the two sharded open devices share: the FRI owner runs the commit phase alone, and every other rank replays the
// transcript from ONE broadcast of (roots, PoW witnesses, folded vector): the number of rounds and every length are known from
// the shapes alone.
class ShardedOpenDevice : public OpenDevice {
  public:
    ~ShardedOpenDevice() override {
        if (op_) msgpu_open_free(op_);
    }
    size_t current_len() override { return cur_len_; }
    // FRI owner only
    Digest commit_round() override {
        Digest d{};
        gpu_check(msgpu_fri_commit_round(op_, d.data()));
        return d;
    }
    void fold(Fp2 beta) override {
        uint64_t b[2] = {beta.c[0].v, beta.c[1].v};
        gpu_check(msgpu_fri_fold(op_, b));
        cur_len_ /= 2;
    }
    void commit_phase(Challenger& ch, size_t stop_len, size_t pow_bits, FriProof& proof) override {
        size_t rounds = 0;
        for (size_t l = cur_len_; l > stop_len; l >>= 1) rounds++;
        const size_t final_len = cur_len_ >> rounds;
        std::vector<u8> blob(rounds * 40 + final_len * 16);
        rs_trace(comm_.rank(), "fri commit phase", rounds);
        if (comm_.rank() == fri_owner_) {
            owner_commit_phase(ch, stop_len, pow_bits, proof);
            if (proof.commit_phase_commits.size() != rounds) throw DistError("fri: internal error, round count");
            for (size_t k = 0; k < rounds; k++) {
                memcpy(blob.data() + 40 * k, proof.commit_phase_commits[k].data(), 32);
                memcpy(blob.data() + 40 * k + 32, &proof.commit_pow_witnesses[k].v, 8);
            }
            gpu_check(msgpu_fri_read_current(op_, (uint64_t*)(blob.data() + rounds * 40)));
        }
        comm_.bcast(blob.data(), blob.size(), fri_owner_);
        if (comm_.rank() != fri_owner_) {
            for (size_t k = 0; k < rounds; k++) {
                Digest d;
                Fp w;
                memcpy(d.data(), blob.data() + 40 * k, 32);
                memcpy(&w.v, blob.data() + 40 * k + 32, 8);
                ch.observe(d);
                proof.commit_phase_commits.push_back(d);
                if (!ch.check_witness(pow_bits, w)) throw DistError("fri: the owner's proof-of-work witness does not verify");
                proof.commit_pow_witnesses.push_back(w);
                betas.push_back(ch.sample_ext());
            }
        }
        cur_len_ = final_len;
        folded_.resize(final_len);
        const uint64_t* f = (const uint64_t*)(blob.data() + rounds * 40);
        for (size_t i = 0; i < final_len; i++) { folded_[i].c[0].v = f[2 * i]; folded_[i].c[1].v = f[2 * i + 1]; }
    }
    std::vector<Fp2> read_current() override { return folded_; }

  protected:
    ShardedOpenDevice(msgpu_ctx* ctx, const CommView& comm, const std::vector<OpenRound>& rounds) : ctx_(ctx), comm_(comm), rounds_(rounds) {}
    // the FRI owner's rounds (the host loop unless overridden)
    virtual void owner_commit_phase(Challenger& ch, size_t stop_len, size_t pow_bits, FriProof& proof) {
        OpenDevice::commit_phase(ch, stop_len, pow_bits, proof);
    }
    msgpu_ctx* ctx_;
    CommView comm_;
    std::vector<OpenRound> rounds_;
    msgpu_open* op_ = nullptr;
    int fri_owner_ = 0;
    unsigned log_max_height_ = 0;
    size_t cur_len_ = 0;
    std::vector<Fp2> folded_;
};

// Pcs::ProverData of a sharded commitment.
struct DistPcsHandle : PcsHandle {
    std::vector<std::pair<size_t, size_t>> shapes;  // every matrix of the commitment: (LDE height, width), commit order
    std::vector<int> owner;                         // rank holding matrix i
    std::vector<int> local_index;                   // index inside `local`, -1 if the matrix lives elsewhere
    PdataPtr local;                                 // this rank's matrices (rows, no tree); null if it has none
    PdataPtr tree;                                  // digest layers, on the tree owner only
    int tree_owner = 0;
    size_t num_matrices() const override { return shapes.size(); }
    size_t matrix_height(size_t i) const override { return shapes[i].first; }
    size_t matrix_width(size_t i) const override { return shapes[i].second; }
    size_t local_max_height() const { return local ? (size_t)msgpu_pdata_max_height(local.get()) : 0; }
    std::vector<size_t> matrices_of(int rank) const {
        std::vector<size_t> v;
        for (size_t i = 0; i < owner.size(); i++)
            if (owner[i] == rank) v.push_back(i);
        return v;
    }
};

// height class -> owner, checked: a class must not be split over ranks
inline std::map<size_t, int, std::greater<size_t>> class_owners(const std::vector<std::pair<size_t, size_t>>& shapes,
                                                                const std::vector<int>& owner) {
    std::map<size_t, int, std::greater<size_t>> cls;
    for (size_t i = 0; i < shapes.size(); i++) {
        auto it = cls.find(shapes[i].first);
        if (it == cls.end()) cls[shapes[i].first] = owner[i];
        else if (it->second != owner[i])
            throw DistError("sharded proof: circuits of one height (2^" + std::to_string(log2_strict(shapes[i].first)) +
                            " LDE rows) must live on one rank");
    }
    return cls;
}

struct DistMatrix {
    size_t height, width;  // of the input (evaluations: trace height; LDEs: LDE height)
    int owner;
    uint64_t* dev;  // on the owner
};

// Pcs::commit / commit_ldes over the ranks. `ldes` (commit_ldes): this rank's LDE buffers in commit order, released to the
// prover data once it has adopted them. `local`: the local part already built from `mats` (msgpu_commit_upload with
// local_only = 1).
inline std::shared_ptr<DistPcsHandle> dist_commit(msgpu_ctx* ctx, const CommView& comm, const std::vector<DistMatrix>& mats, uint32_t log_blowup,
                                                  Digest& root, PdataPtr local = nullptr, std::vector<DevBuf>* ldes = nullptr) {
    auto h = std::make_shared<DistPcsHandle>();
    h->local = std::move(local);
    std::vector<uint64_t*> ptrs;
    std::vector<uint64_t> hs, ws;
    for (auto& m : mats) {
        h->shapes.push_back({ldes ? m.height : (m.height << log_blowup), m.width});
        h->owner.push_back(m.owner);
        if (m.owner == comm.rank()) {
            h->local_index.push_back((int)ptrs.size());
            ptrs.push_back(m.dev);
            hs.push_back(m.height);
            ws.push_back(m.width);
        } else {
            h->local_index.push_back(-1);
        }
    }
    if (mats.empty()) throw DistError("commit: no matrices given");
    auto cls = class_owners(h->shapes, h->owner);
    h->tree_owner = cls.begin()->second;
    if (!h->local && !ptrs.empty()) {
        msgpu_pdata* pd = nullptr;
        gpu_check(msgpu_commit_local_dev(ctx, ptrs.data(), hs.data(), ws.data(), ptrs.size(), log_blowup, ldes ? 1 : 0, &pd));
        h->local.reset(pd);
        // adopted only on success: from here on the handle releases them, and the caller must not -- the arena knows blocks by
        // address only, and a released address may already be live elsewhere
        if (ldes)
            for (auto& b : *ldes) b.release();
    }
    // class digests -> tree owner
    std::vector<uint64_t> class_h;
    std::vector<const uint8_t*> class_ptr;
    std::vector<DevBuf> received;
    auto local_class = [&](size_t height) -> uint8_t* {
        for (uint64_t k = 0; h->local && k < msgpu_pdata_num_classes(h->local.get()); k++) {
            uint64_t lh = 0;
            uint8_t* p = nullptr;
            gpu_check(msgpu_pdata_class_digests(h->local.get(), k, &lh, &p));
            if (lh == height) return p;
        }
        throw DistError("commit: internal error, class digests missing");
    };
    for (auto& kv : cls) {
        size_t height = kv.first;
        int own = kv.second;
        if (own == h->tree_owner) {
            if (comm.rank() == own) { class_h.push_back(height); class_ptr.push_back(local_class(height)); }
            continue;
        }
        if (comm.rank() == own) {
            comm.sendrecv_dev(local_class(height), height * 32, own, h->tree_owner);
        } else if (comm.rank() == h->tree_owner) {
            received.emplace_back(ctx, height * 32);
            comm.sendrecv_dev(received.back().get(), height * 32, own, h->tree_owner);
            class_h.push_back(height);
            class_ptr.push_back((const uint8_t*)received.back().get());
        }
    }
    if (comm.rank() == h->tree_owner) {
        msgpu_pdata* pd = nullptr;
        gpu_check(msgpu_tree_from_digests(ctx, class_h.size(), class_h.data(), class_ptr.data(), &pd, root.data()));
        h->tree.reset(pd);
    }
    received.clear();
    comm.bcast(root.data(), 32, h->tree_owner);
    return h;
}

class DistOpenDevice : public ShardedOpenDevice {
  public:
    DistOpenDevice(msgpu_ctx* ctx, const CommView& comm, const std::vector<OpenRound>& rounds, uint32_t log_blowup)
        : ShardedOpenDevice(ctx, comm, rounds) {
        std::vector<const msgpu_pdata*> pds;
        std::vector<uint64_t> npts, pts;
        std::vector<std::pair<size_t, size_t>> all_shapes;
        std::vector<int> all_owner;
        for (auto& r : rounds) {
            auto* h = dynamic_cast<DistPcsHandle*>(r.data);
            if (!h) throw DistError("open: prover data does not belong to the sharded backend");
            if (r.points.size() != h->shapes.size()) throw DistError("open: one point list per committed matrix expected");
            handles_.push_back(h);
            all_shapes.insert(all_shapes.end(), h->shapes.begin(), h->shapes.end());
            all_owner.insert(all_owner.end(), h->owner.begin(), h->owner.end());
            if (!h->local) continue;
            pds.push_back(h->local.get());
            for (size_t m = 0; m < h->shapes.size(); m++) {
                if (h->local_index[m] < 0) continue;
                npts.push_back(r.points[m].size());
                for (auto& z : r.points[m]) { pts.push_back(z.c[0].v); pts.push_back(z.c[1].v); }
            }
        }
        classes_ = class_owners(all_shapes, all_owner);
        fri_owner_ = classes_.begin()->second;
        log_max_height_ = log2_strict(classes_.begin()->first);
        if (pts.empty()) pts.push_back(0);
        if (!pds.empty()) gpu_check(msgpu_open_begin(ctx_, pds.size(), pds.data(), npts.data(), pts.data(), log_blowup, &op_, &n_local_values_));
    }

    std::vector<OpenedValuesForRound> evaluate() override {
        // global flat layout (round, matrix, point, column); every rank fills the values of its matrices
        std::vector<size_t> len;  // u64 of matrix (r, m), in that order
        size_t total = 0;
        for (size_t r = 0; r < handles_.size(); r++)
            for (size_t m = 0; m < handles_[r]->shapes.size(); m++) {
                len.push_back(2 * rounds_[r].points[m].size() * handles_[r]->shapes[m].second);
                total += len.back();
            }
        std::vector<uint64_t> local(std::max<size_t>(2 * n_local_values_, 1)), mine(std::max<size_t>(total, 1), 0);
        if (op_) gpu_check(msgpu_open_values(op_, local.data()));
        size_t lo = 0, go = 0, i = 0;
        for (size_t r = 0; r < handles_.size(); r++)
            for (size_t m = 0; m < handles_[r]->shapes.size(); m++, go += len[i++])
                if (handles_[r]->owner[m] == comm_.rank()) {
                    memcpy(mine.data() + go, local.data() + lo, len[i] * 8);
                    lo += len[i];
                }
        std::vector<uint64_t> all(mine.size() * comm_.world());
        comm_.allgather(mine.data(), all.data(), mine.size() * 8);
        // every matrix's values from its owner's share
        go = i = 0;
        for (size_t r = 0; r < handles_.size(); r++)
            for (size_t m = 0; m < handles_[r]->shapes.size(); m++, go += len[i++])
                memcpy(mine.data() + go, all.data() + (size_t)handles_[r]->owner[m] * mine.size() + go, len[i] * 8);
        return decode_opened_values(rounds_, mine.data());
    }

    void reduce(Fp2 alpha, unsigned& log_max_height) override {
        uint64_t a[2] = {alpha.c[0].v, alpha.c[1].v}, n_inputs = 0;
        uint32_t lm = 0;
        if (op_) gpu_check(msgpu_open_reduce(op_, a, &n_inputs, &lm));
        // every height class that does not live on the FRI owner travels there (16 B per LDE row), tallest first
        for (auto& kv : classes_) {
            size_t len = kv.first;
            int own = kv.second;
            if (own == fri_owner_) continue;
            if (comm_.rank() == own) {
                uint64_t* p = nullptr;
                for (uint64_t k = 0; k < n_inputs && !p; k++) {
                    uint64_t l = 0;
                    uint64_t* q = nullptr;
                    gpu_check(msgpu_open_input_dev(op_, k, &q, &l));
                    if (l == len) p = q;
                }
                if (!p) throw DistError("open: internal error, reduced openings of a local height class missing");
                comm_.sendrecv_dev(p, len * 16, own, fri_owner_);
            } else if (comm_.rank() == fri_owner_) {
                uint64_t* p = nullptr;
                gpu_check(msgpu_open_add_input(op_, len, &p));
                comm_.sendrecv_dev(p, len * 16, own, fri_owner_);
            }
        }
        cur_len_ = size_t(1) << log_max_height_;
        log_max_height = log_max_height_;
    }

    // What rank `rk` contributes to the query phase, in the order of its msgpu_open_batch_multi call.
    struct Piece {
        enum Kind { Rows, Path, Layer } kind;
        size_t round_or_layer;
        std::vector<size_t> mats;  // Rows: global matrix indices of the round held by the rank
        TreeShape shape;
    };
    std::vector<Piece> pieces_of(int rk, const std::vector<unsigned>& round_shifts, size_t n_layers) const {
        std::vector<Piece> v;
        for (size_t r = 0; r < handles_.size(); r++) {
            auto mine = handles_[r]->matrices_of(rk);
            if (!mine.empty()) {
                TreeShape s;
                for (size_t m : mine) s.widths.push_back(handles_[r]->shapes[m].second);
                v.push_back(Piece{Piece::Rows, r, mine, s});
            }
            if (handles_[r]->tree_owner == rk) v.push_back(Piece{Piece::Path, r, {}, TreeShape{{}, (size_t)(log_max_height_ - round_shifts[r])}});
        }
        if (rk == fri_owner_)
            for (size_t k = 0; k < n_layers; k++) v.push_back(Piece{Piece::Layer, k, {}, TreeShape{{4}, (size_t)(log_max_height_ - k - 1)}});
        return v;
    }

    void open_queries(const std::vector<size_t>& indices, const std::vector<unsigned>& round_shifts, size_t n_layers,
                      std::vector<std::vector<BatchOpening>>& rounds_out, std::vector<std::vector<BatchOpening>>& layers_out) override {
        const size_t n = indices.size();
        const bool trace = getenv("MSH_TRACE") != nullptr;
        auto tq0 = std::chrono::steady_clock::now();
        auto lapq = [&](const char* what) {
            auto t1 = std::chrono::steady_clock::now();
            if (trace) fprintf(stderr, "[msh] rank %d queries/%-12s %8.3f ms\n", comm_.rank(), what, std::chrono::duration<double, std::milli>(t1 - tq0).count());
            tq0 = t1;
        };
        // this rank's share in one launch
        std::vector<const msgpu_pdata*> trees;
        std::vector<uint32_t> shifts;
        std::vector<TreeShape> shapes;
        for (auto& pc : pieces_of(comm_.rank(), round_shifts, n_layers)) {
            if (pc.kind == Piece::Rows) {
                trees.push_back(handles_[pc.round_or_layer]->local.get());
                shifts.push_back((uint32_t)(log_max_height_ - log2_strict(handles_[pc.round_or_layer]->local_max_height())));
            } else if (pc.kind == Piece::Path) {
                trees.push_back(handles_[pc.round_or_layer]->tree.get());
                shifts.push_back(round_shifts[pc.round_or_layer]);
            } else {
                trees.push_back(fri_layer(op_, pc.round_or_layer));
                shifts.push_back((uint32_t)(pc.round_or_layer + 1));
            }
            shapes.push_back(pc.shape);
        }
        std::vector<u8> blob = open_batch_multi(ctx_, trees, shifts, shapes, indices);
        lapq("local_open");
        std::vector<std::vector<u8>> all = comm_.allgather_var(blob);
        lapq("allgather");

        rounds_out.assign(handles_.size(), std::vector<BatchOpening>(n));
        layers_out.assign(n_layers, std::vector<BatchOpening>(n));
        for (size_t r = 0; r < handles_.size(); r++)
            for (size_t q = 0; q < n; q++) rounds_out[r][q].opened_values.resize(handles_[r]->shapes.size());
        for (int rk = 0; rk < comm_.world(); rk++) {
            auto pcs = pieces_of(rk, round_shifts, n_layers);
            shapes.clear();
            for (auto& pc : pcs) shapes.push_back(pc.shape);
            if (all[rk].size() != batch_bytes(shapes, n)) throw DistError("open: a rank sent a query share of unexpected size");
            auto got = decode_batch_openings(shapes, n, all[rk]);
            for (size_t i = 0; i < pcs.size(); i++)
                for (size_t q = 0; q < n; q++) {
                    const Piece& pc = pcs[i];
                    if (pc.kind == Piece::Layer) {
                        layers_out[pc.round_or_layer][q] = std::move(got[i][q]);
                        continue;
                    }
                    BatchOpening& bo = rounds_out[pc.round_or_layer][q];
                    for (size_t j = 0; j < pc.mats.size(); j++) bo.opened_values[pc.mats[j]] = std::move(got[i][q].opened_values[j]);
                    if (pc.kind == Piece::Path) bo.opening_proof = std::move(got[i][q].opening_proof);
                }
        }
        lapq("assemble");
    }

  private:
    uint64_t n_local_values_ = 0;
    std::vector<DistPcsHandle*> handles_;
    std::map<size_t, int, std::greater<size_t>> classes_;
};

class DistGpuBackend : public ShardedBackend {
  public:
    // owner[ci] = rank that holds circuit ci
    DistGpuBackend(msgpu_ctx* ctx, const SystemShape& shape, const msh_comm& comm, const std::vector<int>& owner)
        : ShardedBackend(ctx, shape, comm), owner_(owner) {
        if (owner_.size() != shape.circuits.size()) throw DistError("sharded prover: one owner per circuit expected");
        for (int o : owner_)
            if (o < 0 || o >= comm_.world()) throw DistError("sharded prover: owner rank out of range");
    }

    // System::new: the preprocessed commitment over every circuit that has a preprocessed trace (src/system.rs:180-196)
    PcsHandlePtr commit(const std::vector<const Matrix*>& evals, Digest& root) override {
        std::vector<DistMatrix> mats;
        std::vector<DevBuf> up;
        size_t k = 0;
        for (size_t ci = 0; ci < shape_.circuits.size(); ci++) {
            if (!shape_.circuits[ci].has_preprocessed) continue;
            if (k >= evals.size()) throw DistError("commit: preprocessed matrix list does not match the system");
            const Matrix* m = evals[k++];
            DistMatrix dm{m->height(), m->width, owner_[ci], nullptr};
            if (owner_[ci] == comm_.rank()) {
                up.push_back(upload((const uint64_t*)m->values.data(), m->values.size()));
                dm.dev = up.back().get();
            }
            mats.push_back(dm);
        }
        return dist_commit(ctx_, comm_, mats, (uint32_t)shape_.log_blowup(), root);
    }

    PcsHandlePtr commit_stage1(const std::vector<size_t>& circuits, const std::vector<MatrixView>& traces, Digest& root) override {
        end_proof();
        active_ = circuits;
        std::vector<DistMatrix> mats;
        std::vector<const uint64_t*> ptrs;
        std::vector<uint64_t> hs, ws;
        std::vector<size_t> local_pos;
        for (size_t p = 0; p < circuits.size(); p++) {
            const MatrixView& m = traces[p];
            mats.push_back(DistMatrix{m.height(), m.width, owner_[circuits[p]], nullptr});
            trace_rows_.push_back(m.height());
            if (mats.back().owner != comm_.rank()) continue;
            if (!m.data) throw DistError("sharded prover: the trace of a circuit this rank owns is missing");
            ptrs.push_back((const uint64_t*)m.data);
            hs.push_back(m.height());
            ws.push_back(m.width);
            local_pos.push_back(p);
        }
        // The claims are handled by the rank with the least trace data. (Every rank doing it put N copies of the claims on the
        // host's PCIe.)
        {
            std::vector<uint64_t> load(comm_.world(), 0);
            for (auto& m : mats) load[m.owner] += (uint64_t)m.height * m.width;
            claims_rank_ = 0;
            for (int r = 0; r < comm_.world(); r++)
                if (load[r] <= load[claims_rank_]) claims_rank_ = r;
            if (comm_.rank() != claims_rank_) announced_ = ClaimsView();
        }
        trace_dev_.resize(circuits.size());
        PdataPtr local;
        if (!ptrs.empty()) {
            // this rank's traces cross PCIe on the copy stream while the earlier ones are extended; the claims follow them
            msgpu_upload* up = nullptr;
            gpu_check(msgpu_upload_begin(ctx_, ptrs.data(), hs.data(), ws.data(), ptrs.size(), &up));
            std::unique_ptr<msgpu_upload, void (*)(msgpu_upload*)> pending(up, msgpu_upload_free);
            prefetch_announced_claims();
            std::vector<uint64_t*> kept(ptrs.size(), nullptr);
            msgpu_pdata* pd = nullptr;
            // takes the upload on every path; the kept inputs are ours only on success
            gpu_check(msgpu_commit_upload(pending.release(), (uint32_t)shape_.log_blowup(), 1, kept.data(), 1, &pd, nullptr));
            local.reset(pd);
            for (size_t k = 0; k < kept.size(); k++) {
                trace_dev_[local_pos[k]] = DevBuf(ctx_, kept[k]);
                mats[local_pos[k]].dev = kept[k];
            }
        } else {
            prefetch_announced_claims();
        }
        return dist_commit(ctx_, comm_, mats, (uint32_t)shape_.log_blowup(), root, std::move(local));
    }

    PcsHandlePtr commit_stage2(Fp2 beta, Fp2 gamma, Fp2 acc, std::vector<Fp2>& intermediate, Digest& root) override {
        uint64_t b[2] = {beta.c[0].v, beta.c[1].v}, g[2] = {gamma.c[0].v, gamma.c[1].v};
        std::vector<DistMatrix> mats;
        std::vector<uint64_t> sums(2 * active_.size(), 0);
        std::vector<DevBuf> s2;  // scratch
        for (size_t p = 0; p < active_.size(); p++) {
            const Circuit& c = shape_.circuits[active_[p]];
            uint64_t rows = trace_rows_[p];
            DistMatrix dm{rows, c.stage_2_width, owner_[active_[p]], nullptr};
            if (dm.owner == comm_.rank()) {
                s2.emplace_back(ctx_, rows * c.stage_2_width * 8);
                dm.dev = s2.back().get();
                gpu_check(msgpu_stage2_trace(ctx_, programs_[active_[p]], pre_dev_[active_[p]].get(), trace_dev_[p].get(), rows, b, g, dm.dev,
                                             &sums[2 * p]));
            }
            mats.push_back(dm);
        }
        // chain the per-circuit sums of all ranks (src/lookup.rs:530-543 runs this chain serially over the circuits)
        std::vector<uint64_t> all(sums.size() * comm_.world());
        comm_.allgather(sums.data(), all.data(), sums.size() * 8);
        intermediate.clear();
        for (size_t p = 0; p < active_.size(); p++) {
            const uint64_t* s = all.data() + (size_t)owner_[active_[p]] * sums.size() + 2 * p;
            acc += Fp2(Fp(s[0]), Fp(s[1]));
            intermediate.push_back(acc);
        }
        auto h = dist_commit(ctx_, comm_, mats, (uint32_t)shape_.log_blowup(), root);
        s2.clear();
        trace_dev_.clear();
        return h;
    }

    PcsHandlePtr commit_quotient(const std::vector<QuotientJob>& jobs, PcsHandle* pre, PcsHandle* s1, PcsHandle* s2, Fp2 alpha,
                                 Digest& root) override {
        auto* h1 = dynamic_cast<DistPcsHandle*>(s1);
        auto* h2 = dynamic_cast<DistPcsHandle*>(s2);
        auto* hp = pre ? dynamic_cast<DistPcsHandle*>(pre) : nullptr;
        if (!h1 || !h2 || (pre && !hp)) throw DistError("quotient: prover data does not belong to the sharded backend");
        uint64_t a[2] = {alpha.c[0].v, alpha.c[1].v};
        uint32_t lb = (uint32_t)shape_.log_blowup();
        std::vector<DistMatrix> mats;
        std::vector<DevBuf> ldes;
        for (auto& j : jobs) {
            DistMatrix dm{(size_t)1 << (j.log_degree + lb), (size_t)2 << j.log_quotient_degree, owner_[j.circuit], nullptr};
            if (dm.owner == comm_.rank()) {
                uint64_t pub[8];
                for (int k = 0; k < 8; k++) pub[k] = j.publics[k].v;
                const msgpu_pdata* ppd = nullptr;
                uint64_t pidx = 0;
                if (j.preprocessed_idx >= 0 && hp) {
                    ppd = hp->local.get();
                    pidx = (uint64_t)hp->local_index[j.preprocessed_idx];
                }
                gpu_check(msgpu_quotient(ctx_, programs_[j.circuit], ppd, pidx, h1->local.get(), (uint64_t)h1->local_index[j.pos], h2->local.get(),
                                         (uint64_t)h2->local_index[j.pos], j.log_degree, j.log_quotient_degree, lb, pub, a, &dm.dev, nullptr));
                ldes.emplace_back(ctx_, dm.dev);
            }
            mats.push_back(dm);
        }
        return dist_commit(ctx_, comm_, mats, lb, root, nullptr, &ldes);
    }

    std::unique_ptr<OpenDevice> open_begin(const std::vector<OpenRound>& rounds) override {
        return std::make_unique<DistOpenDevice>(ctx_, comm_, rounds, (uint32_t)shape_.log_blowup());
    }

  private:
    std::vector<int> owner_;
};

}  // namespace msh
