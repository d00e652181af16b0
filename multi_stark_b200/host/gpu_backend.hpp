// ProverBackend over the libmsgpu C ABI (include/msgpu.h): what a Rust `GpuFriPcs` + the prover.rs hook
// would call (INTEGRATION.md). All matrices stay resident in HBM between the LDE, Merkle, quotient and opening
// stages; the host sees roots, opened values, the final polynomial and the query openings only.
#pragma once
#include "prover.hpp"
#include <cstdlib>
#include <cstring>
#include <memory>
#include "program.hpp"
#include "../../include/msgpu.h"

namespace msh {

struct GpuError : std::runtime_error {
    using std::runtime_error::runtime_error;
};
inline void gpu_check(int code) {
    if (code != 0) throw GpuError(std::string("libmsgpu: ") + msgpu_last_error());
}

// A device buffer from the context's arena, released with it. Move-only. The adopting constructor takes over a buffer the
// library handed out (the kept inputs of msgpu_commit_upload, the LDE of msgpu_quotient / msgpu_quotient_finish); release()
// gives one up to a call that adopts it, once that call has succeeded.
class DevBuf {
  public:
    DevBuf() = default;
    DevBuf(msgpu_ctx* ctx, size_t bytes) : ctx_(ctx) {
        void* p = nullptr;
        gpu_check(msgpu_malloc(ctx_, std::max<size_t>(bytes, 8), &p));
        p_ = (uint64_t*)p;
    }
    DevBuf(msgpu_ctx* ctx, uint64_t* adopted) : ctx_(ctx), p_(adopted) {}
    DevBuf(DevBuf&& o) noexcept : ctx_(o.ctx_), p_(o.release()) {}
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) {
            reset();
            ctx_ = o.ctx_;
            p_ = o.release();
        }
        return *this;
    }
    ~DevBuf() { reset(); }
    void reset() {
        if (p_) msgpu_free(ctx_, p_);
        p_ = nullptr;
    }
    uint64_t* release() {
        uint64_t* p = p_;
        p_ = nullptr;
        return p;
    }
    uint64_t* get() const { return p_; }

  private:
    msgpu_ctx* ctx_ = nullptr;
    uint64_t* p_ = nullptr;
};

inline std::vector<uint64_t*> raw_ptrs(const std::vector<DevBuf>& v) {
    std::vector<uint64_t*> out;
    for (auto& b : v) out.push_back(b.get());
    return out;
}

struct PdataFree {
    void operator()(msgpu_pdata* pd) const { msgpu_pdata_free(pd); }
};
using PdataPtr = std::unique_ptr<msgpu_pdata, PdataFree>;

struct GpuPcsHandle : PcsHandle {
    PdataPtr owned;  // empty when the handle borrows the caller's prover data (msh_pcs_open)
    const msgpu_pdata* pd = nullptr;
    std::vector<std::pair<size_t, size_t>> shapes;
    explicit GpuPcsHandle(const msgpu_pdata* p) : pd(p) {
        for (uint64_t i = 0; i < msgpu_pdata_num_matrices(pd); i++) {
            uint64_t r = 0, c = 0;
            gpu_check(msgpu_pdata_matrix(pd, i, nullptr, &r, &c));
            shapes.push_back({(size_t)r, (size_t)c});
        }
    }
    explicit GpuPcsHandle(PdataPtr p) : GpuPcsHandle(p.get()) { owned = std::move(p); }
    size_t num_matrices() const override { return shapes.size(); }
    size_t matrix_height(size_t i) const override { return shapes[i].first; }
    size_t matrix_width(size_t i) const override { return shapes[i].second; }
};

// msgpu_open_values output -- (round, matrix, point, column), 2 u64 per value -- as [round][matrix][point][column]
inline std::vector<OpenedValuesForRound> decode_opened_values(const std::vector<OpenRound>& rounds, const uint64_t* flat) {
    std::vector<OpenedValuesForRound> out(rounds.size());
    size_t o = 0;
    for (size_t r = 0; r < rounds.size(); r++) {
        out[r].resize(rounds[r].points.size());
        for (size_t m = 0; m < rounds[r].points.size(); m++) {
            out[r][m].resize(rounds[r].points[m].size());
            for (auto& pv : out[r][m]) {
                pv.resize(rounds[r].data->matrix_width(m));
                for (auto& v : pv) { v.c[0].v = flat[o++]; v.c[1].v = flat[o++]; }
            }
        }
    }
    return out;
}

// One tree of an msgpu_open_batch[_multi] result: the widths of its matrices and the sibling digests per query.
struct TreeShape {
    std::vector<size_t> widths;
    size_t depth = 0;
};
inline TreeShape tree_shape(const msgpu_pdata* pd) {
    TreeShape s;
    size_t maxh = 0;
    for (uint64_t i = 0; i < msgpu_pdata_num_matrices(pd); i++) {
        uint64_t r = 0, c = 0;
        gpu_check(msgpu_pdata_matrix(pd, i, nullptr, &r, &c));
        s.widths.push_back((size_t)c);
        maxh = std::max(maxh, (size_t)r);
    }
    s.depth = log2_strict(maxh);
    return s;
}
// An msgpu_open_batch_multi result for n queries in one buffer: every tree's rows (8 bytes a value), then every tree's paths
inline size_t batch_row_bytes(const std::vector<TreeShape>& trees, size_t n) {
    size_t b = 0;
    for (auto& t : trees)
        for (size_t w : t.widths) b += n * w * 8;
    return b;
}
inline size_t batch_bytes(const std::vector<TreeShape>& trees, size_t n) {
    size_t b = batch_row_bytes(trees, n);
    for (auto& t : trees) b += n * t.depth * 32;
    return b;
}
// tree t opened at indices[q] >> shifts[t]
inline std::vector<u8> open_batch_multi(msgpu_ctx* ctx, const std::vector<const msgpu_pdata*>& trees, const std::vector<uint32_t>& shifts,
                                        const std::vector<TreeShape>& shapes, const std::vector<size_t>& indices) {
    const size_t n = indices.size(), rb = batch_row_bytes(shapes, n), total = batch_bytes(shapes, n);
    std::vector<u8> out(std::max<size_t>(total, 8));
    if (!trees.empty()) {
        std::vector<uint64_t> idx(indices.begin(), indices.end());
        gpu_check(msgpu_open_batch_multi(ctx, trees.data(), shifts.data(), trees.size(), idx.data(), n, (uint64_t*)out.data(), out.data() + rb));
    }
    out.resize(total);
    return out;
}
// [tree][query] from such a buffer
inline std::vector<std::vector<BatchOpening>> decode_batch_openings(const std::vector<TreeShape>& shapes, size_t n, const std::vector<u8>& buf) {
    if (buf.size() != batch_bytes(shapes, n)) throw GpuError("open: internal error, batch opening size");
    const u8* ro = buf.data();
    const u8* po = buf.data() + batch_row_bytes(shapes, n);
    std::vector<std::vector<BatchOpening>> out(shapes.size(), std::vector<BatchOpening>(n));
    for (size_t t = 0; t < shapes.size(); t++)
        for (auto& bo : out[t]) {
            for (size_t w : shapes[t].widths) {
                std::vector<Fp> row(w);
                if (w) memcpy(row.data(), ro, w * 8);
                ro += w * 8;
                bo.opened_values.push_back(std::move(row));
            }
            bo.opening_proof.resize(shapes[t].depth);
            for (auto& sib : bo.opening_proof) {
                memcpy(sib.data(), po, 32);
                po += 32;
            }
        }
    return out;
}

inline const msgpu_pdata* fri_layer(msgpu_open* op, size_t k) {
    const msgpu_pdata* pd = msgpu_fri_layer_pdata(op, k);
    if (!pd) throw GpuError("open: no such commit-phase layer");
    return pd;
}

// p3-fri `commit_phase` with the transcript on the device (no root read-back per round); the host challenger replays the rounds
// afterwards and every beta is compared. Returns false, having done nothing, where that path does not apply: a proof of work to
// grind, a challenger buffer the device transcript does not take (empty or over 960 bytes), more than 64 rounds or none.
inline bool fri_commit_phase_on_device(msgpu_open* op, size_t cur_len, Challenger& ch, size_t stop_len, size_t pow_bits, FriProof& proof,
                                       std::vector<Fp2>& betas) {
    const std::vector<u8>& buf = ch.input_buffer();
    size_t rounds = 0;
    for (size_t l = cur_len; l > stop_len; l >>= 1) rounds++;
    if (pow_bits != 0 || buf.empty() || buf.size() > 960 || rounds == 0 || rounds > 64) return false;
    uint8_t roots[64 * 32];
    uint64_t bt[64 * 2], n = 0;
    gpu_check(msgpu_fri_commit_phase(op, buf.data(), buf.size(), stop_len, 64, roots, bt, &n));
    for (uint64_t k = 0; k < n; k++) {
        Digest commit;
        memcpy(commit.data(), roots + 32 * k, 32);
        ch.observe(commit);
        proof.commit_phase_commits.push_back(commit);
        proof.commit_pow_witnesses.push_back(ch.grind(0));
        Fp2 beta = ch.sample_ext();
        if (beta.c[0].v != bt[2 * k] || beta.c[1].v != bt[2 * k + 1])
            throw GpuError("fri: the device transcript and the host challenger disagree on a folding challenge");
        betas.push_back(beta);
    }
    return true;
}

class GpuOpenDevice : public OpenDevice {
  public:
    GpuOpenDevice(msgpu_ctx* ctx, const std::vector<OpenRound>& rounds, uint32_t log_blowup) : ctx_(ctx), rounds_(rounds) {
        std::vector<uint64_t> npts, pts;
        for (auto& r : rounds) {
            auto* h = dynamic_cast<GpuPcsHandle*>(r.data);
            if (!h) throw GpuError("open: prover data does not belong to the GPU backend");
            pds_.push_back(h->pd);
            if (r.points.size() != h->shapes.size()) throw GpuError("open: one point list per committed matrix expected");
            for (auto& mp : r.points) {
                npts.push_back(mp.size());
                for (auto& z : mp) { pts.push_back(z.c[0].v); pts.push_back(z.c[1].v); }
            }
        }
        if (pts.empty()) pts.push_back(0);
        gpu_check(msgpu_open_begin(ctx_, pds_.size(), pds_.data(), npts.data(), pts.data(), log_blowup, &op_, &n_values_));
    }
    ~GpuOpenDevice() override { msgpu_open_free(op_); }

    std::vector<OpenedValuesForRound> evaluate() override {
        std::vector<uint64_t> flat(std::max<size_t>(2 * n_values_, 1));
        gpu_check(msgpu_open_values(op_, flat.data()));
        return decode_opened_values(rounds_, flat.data());
    }
    void reduce(Fp2 alpha, unsigned& log_max_height) override {
        uint64_t a[2] = {alpha.c[0].v, alpha.c[1].v}, n = 0;
        uint32_t lm = 0;
        gpu_check(msgpu_open_reduce(op_, a, &n, &lm));
        log_max_height = lm;
    }
    size_t current_len() override {
        uint64_t len = 0;
        gpu_check(msgpu_fri_current_len(op_, &len));
        return (size_t)len;
    }
    Digest commit_round() override {
        Digest d;
        gpu_check(msgpu_fri_commit_round(op_, d.data()));
        return d;
    }
    void fold(Fp2 beta) override {
        uint64_t b[2] = {beta.c[0].v, beta.c[1].v};
        gpu_check(msgpu_fri_fold(op_, b));
    }
    void commit_phase(Challenger& ch, size_t stop_len, size_t pow_bits, FriProof& proof) override {
        if (!fri_commit_phase_on_device(op_, current_len(), ch, stop_len, pow_bits, proof, betas)) OpenDevice::commit_phase(ch, stop_len, pow_bits, proof);
    }
    std::vector<Fp2> read_current() override {
        size_t len = current_len();
        std::vector<uint64_t> flat(2 * len);
        gpu_check(msgpu_fri_read_current(op_, flat.data()));
        std::vector<Fp2> out(len);
        for (size_t i = 0; i < len; i++) { out[i].c[0].v = flat[2 * i]; out[i].c[1].v = flat[2 * i + 1]; }
        return out;
    }

    // every round and every commit-phase layer in one launch
    void open_queries(const std::vector<size_t>& indices, const std::vector<unsigned>& round_shifts, size_t n_layers,
                      std::vector<std::vector<BatchOpening>>& rounds_out, std::vector<std::vector<BatchOpening>>& layers_out) override {
        std::vector<const msgpu_pdata*> trees(pds_.begin(), pds_.end());
        std::vector<uint32_t> shifts(round_shifts.begin(), round_shifts.end());
        for (size_t k = 0; k < n_layers; k++) {
            trees.push_back(fri_layer(op_, k));
            shifts.push_back((uint32_t)(k + 1));
        }
        std::vector<TreeShape> shapes;
        for (auto* t : trees) shapes.push_back(tree_shape(t));
        auto all = decode_batch_openings(shapes, indices.size(), open_batch_multi(ctx_, trees, shifts, shapes, indices));
        auto split = all.begin() + (ptrdiff_t)round_shifts.size();
        rounds_out.assign(std::make_move_iterator(all.begin()), std::make_move_iterator(split));
        layers_out.assign(std::make_move_iterator(split), std::make_move_iterator(all.end()));
    }

  private:
    msgpu_ctx* ctx_;
    msgpu_open* op_ = nullptr;
    uint64_t n_values_ = 0;
    std::vector<OpenRound> rounds_;
    std::vector<const msgpu_pdata*> pds_;
};

class GpuBackend : public ProverBackend {
  public:
    GpuBackend(msgpu_ctx* ctx, const SystemShape& shape) : ctx_(ctx), shape_(shape) {
        for (auto& c : shape_.circuits) {
            GraphDesc d;
            d.build(c.graph, c.preprocessed_width, c.main_width, c.stage_2_width);
            msgpu_program* p = nullptr;
            gpu_check(msgpu_program_create(ctx_, &d.desc, &p));
            programs_.push_back(p);
            // the preprocessed trace in natural order stays on the device for the stage-2 construction
            if (c.has_preprocessed && !c.preprocessed.values.empty())
                pre_dev_.push_back(upload((const uint64_t*)c.preprocessed.values.data(), c.preprocessed.values.size()));
            else
                pre_dev_.emplace_back();
        }
    }
    ~GpuBackend() override {
        end_proof();
        for (auto* p : programs_) msgpu_program_free(p);
    }

    PcsHandlePtr commit(const std::vector<const Matrix*>& evals, Digest& root) override {
        std::vector<const uint64_t*> ptrs;
        std::vector<uint64_t> hs, ws;
        for (auto* m : evals) { ptrs.push_back((const uint64_t*)m->values.data()); hs.push_back(m->height()); ws.push_back(m->width); }
        msgpu_pdata* pd = nullptr;
        gpu_check(msgpu_commit(ctx_, ptrs.data(), hs.data(), ws.data(), evals.size(), (uint32_t)shape_.log_blowup(), &pd, root.data()));
        return std::make_shared<GpuPcsHandle>(PdataPtr(pd));
    }

    PcsHandlePtr commit_stage1(const std::vector<size_t>& circuits, const std::vector<MatrixView>& traces, Digest& root) override {
        end_proof();
        active_ = circuits;
        std::vector<const uint64_t*> ptrs;
        std::vector<uint64_t> hs, ws;
        for (auto& m : traces) {
            ptrs.push_back((const uint64_t*)m.data);
            hs.push_back(m.height());
            ws.push_back(m.width);
            trace_rows_.push_back(m.height());
        }
        // uploads on the copy stream (trace i + 1 crosses PCIe while trace i is extended), the claims queued right behind them
        msgpu_upload* up = nullptr;
        gpu_check(msgpu_upload_begin(ctx_, ptrs.data(), hs.data(), ws.data(), traces.size(), &up));
        std::unique_ptr<msgpu_upload, void (*)(msgpu_upload*)> pending(up, msgpu_upload_free);
        prefetch_announced_claims();
        std::vector<uint64_t*> kept(traces.size(), nullptr);
        msgpu_pdata* pd = nullptr;
        // takes the upload on every path; the kept inputs are ours only on success
        gpu_check(msgpu_commit_upload(pending.release(), (uint32_t)shape_.log_blowup(), 1, kept.data(), 0, &pd, root.data()));
        PdataPtr owned(pd);
        for (auto* k : kept) trace_dev_.emplace_back(ctx_, k);
        return std::make_shared<GpuPcsHandle>(std::move(owned));
    }

    void announce_claims(const ClaimsView& claims) override { announced_ = claims; }

    bool observe_claims(Challenger& ch, const ClaimsView& claims) override {
        Digest d;
        if (!claims_transcript_digest(ch.input_buffer(), claims, d)) return false;
        ch.set_flushed(d);
        return true;
    }

    Fp2 claims_accumulator(const ClaimsView& claims, Fp2 beta, Fp2 gamma) override {
        Fp2 acc = Fp2::zero();
        uint64_t b[2] = {beta.c[0].v, beta.c[1].v}, g[2] = {gamma.c[0].v, gamma.c[1].v};
        if (claims_dev_) {  // already resident (observe_claims)
            uint64_t out[2];
            gpu_check(msgpu_claims_accumulate(claims_dev_, b, g, out));
            drop_claims();
            return Fp2(Fp(out[0]), Fp(out[1]));
        }
        // the C ABI takes claims of one length per call; group consecutive claims of equal length
        size_t i = 0;
        while (i < claims.size()) {
            size_t len = claims.len(i), j = i;
            while (j < claims.size() && claims.len(j) == len) j++;
            uint64_t out[2];
            gpu_check(msgpu_claims_accumulator(ctx_, (const uint64_t*)claims.at(i), j - i, len, b, g, out));
            acc += Fp2(Fp(out[0]), Fp(out[1]));
            i = j;
        }
        return acc;
    }

    Challenger::BigHash big_hash() override {
        msgpu_ctx* ctx = ctx_;
        return [ctx](const u8* data, size_t n) {
            Digest d;
            gpu_check(msgpu_blake3_hash(ctx, data, n, d.data()));
            return d;
        };
    }

    PcsHandlePtr commit_stage2(Fp2 beta, Fp2 gamma, Fp2 acc, std::vector<Fp2>& intermediate, Digest& root) override {
        uint64_t b[2] = {beta.c[0].v, beta.c[1].v}, g[2] = {gamma.c[0].v, gamma.c[1].v};
        std::vector<DevBuf> s2;  // scratch, released when this returns or throws
        std::vector<uint64_t> hs, ws;
        intermediate.clear();
        for (size_t p = 0; p < active_.size(); p++) {
            const Circuit& c = shape_.circuits[active_[p]];
            uint64_t rows = trace_rows_[p];
            s2.emplace_back(ctx_, rows * c.stage_2_width * 8);
            uint64_t local[2] = {0, 0};
            gpu_check(msgpu_stage2_trace(ctx_, programs_[active_[p]], pre_dev_[active_[p]].get(), trace_dev_[p].get(), rows, b, g, s2.back().get(), local));
            acc += Fp2(Fp(local[0]), Fp(local[1]));
            intermediate.push_back(acc);
            hs.push_back(rows);
            ws.push_back(c.stage_2_width);
        }
        msgpu_pdata* pd = nullptr;
        gpu_check(msgpu_commit_dev(ctx_, raw_ptrs(s2).data(), hs.data(), ws.data(), s2.size(), (uint32_t)shape_.log_blowup(), &pd, root.data()));
        PdataPtr owned(pd);
        trace_dev_.clear();  // the natural-order traces are not needed any more
        return std::make_shared<GpuPcsHandle>(std::move(owned));
    }

    PcsHandlePtr commit_quotient(const std::vector<QuotientJob>& jobs, PcsHandle* pre, PcsHandle* s1, PcsHandle* s2, Fp2 alpha,
                                 Digest& root) override {
        auto* h1 = dynamic_cast<GpuPcsHandle*>(s1);
        auto* h2 = dynamic_cast<GpuPcsHandle*>(s2);
        auto* hp = pre ? dynamic_cast<GpuPcsHandle*>(pre) : nullptr;
        uint64_t a[2] = {alpha.c[0].v, alpha.c[1].v};
        std::vector<DevBuf> ldes;
        std::vector<uint64_t> hs, ws;
        uint32_t lb = (uint32_t)shape_.log_blowup();
        for (auto& j : jobs) {
            uint64_t pub[8];
            for (int k = 0; k < 8; k++) pub[k] = j.publics[k].v;
            uint64_t* lde = nullptr;
            gpu_check(msgpu_quotient(ctx_, programs_[j.circuit], j.preprocessed_idx >= 0 && hp ? hp->pd : nullptr,
                                     j.preprocessed_idx >= 0 ? (uint64_t)j.preprocessed_idx : 0, h1->pd, j.pos, h2->pd, j.pos, j.log_degree,
                                     j.log_quotient_degree, lb, pub, a, &lde, nullptr));
            ldes.emplace_back(ctx_, lde);
            hs.push_back((uint64_t)1 << (j.log_degree + lb));
            ws.push_back((uint64_t)2 << j.log_quotient_degree);
        }
        msgpu_pdata* pd = nullptr;
        gpu_check(msgpu_commit_ldes_dev(ctx_, raw_ptrs(ldes).data(), hs.data(), ws.data(), ldes.size(), 1, &pd, root.data()));
        for (auto& l : ldes) l.release();  // adopted by the prover data
        return std::make_shared<GpuPcsHandle>(PdataPtr(pd));
    }

    std::unique_ptr<OpenDevice> open_begin(const std::vector<OpenRound>& rounds) override {
        return std::make_unique<GpuOpenDevice>(ctx_, rounds, (uint32_t)shape_.log_blowup());
    }

    void end_proof() override {
        drop_claims();
        trace_dev_.clear();
        trace_rows_.clear();
        active_.clear();
    }

  protected:  // the sharded backend (dist_backend.hpp) reuses the per-circuit state
    // true if the claim set is large and uniform (same rule on every rank: it depends on the shape only)
    static bool claims_on_device(const ClaimsView& claims) {
        size_t len = claims.uniform_len();
        return len != 0 && claims.size() * len >= 4096;
    }
    // BLAKE3(prefix || length-prefixed claims) on the device (false = small or ragged set: the host loop is cheaper; the
    // ABI's precondition is then checked here)
    bool claims_transcript_digest(const std::vector<u8>& prefix, const ClaimsView& claims, Digest& d) {
        if (!claims_on_device(claims)) {
            size_t total = claims.total();
            for (size_t k = 0; k < total; k++)
                if (claims.values[k].v >= GL_P) throw GpuError("claim value is not canonical");
            return false;
        }
        size_t len = claims.uniform_len();
        if (claims_dev_ && prefetched_from_ == (const void*)claims.at(0) && prefetched_n_ == claims.size() && prefetched_len_ == len) {
            gpu_check(msgpu_claims_digest(claims_dev_, prefix.data(), prefix.size(), d.data()));
        } else {
            drop_claims();
            gpu_check(msgpu_claims_upload(ctx_, (const uint64_t*)claims.at(0), claims.size(), len, prefix.data(), prefix.size(), &claims_dev_,
                                          d.data()));
        }
        prefetched_from_ = nullptr;
        return true;
    }
    // H2D copy + check that every value is canonical (the ABI's precondition, verified on the device)
    DevBuf upload(const uint64_t* src, size_t n) {
        DevBuf d(ctx_, n * 8);
        if (n) gpu_check(msgpu_upload_canonical(ctx_, d.get(), src, n));
        return d;
    }
    void drop_claims() {
        if (claims_dev_) msgpu_claims_free(claims_dev_);
        claims_dev_ = nullptr;
        prefetched_from_ = nullptr;
    }
    // same size rule as observe_claims: small or ragged claim sets stay on the host
    void prefetch_announced_claims() {
        ClaimsView cl = announced_;
        announced_ = ClaimsView();
        size_t len = cl.uniform_len();
        if (len == 0 || cl.size() * len < 4096) return;
        drop_claims();
        gpu_check(msgpu_claims_prefetch(ctx_, (const uint64_t*)cl.at(0), cl.size(), len, &claims_dev_));
        prefetched_from_ = (const void*)cl.at(0);
        prefetched_n_ = cl.size();
        prefetched_len_ = len;
    }
    ClaimsView announced_;
    const void* prefetched_from_ = nullptr;
    size_t prefetched_n_ = 0, prefetched_len_ = 0;
    msgpu_ctx* ctx_;
    msgpu_claims* claims_dev_ = nullptr;
    const SystemShape& shape_;
    std::vector<msgpu_program*> programs_;
    std::vector<DevBuf> pre_dev_;
    std::vector<size_t> active_;
    std::vector<DevBuf> trace_dev_;
    std::vector<uint64_t> trace_rows_;
};

}  // namespace msh
