// ORACLE (test infrastructure, not product code): CPU restatement of the PCS the reference configures at
// src/types.rs:85,209-223 -- `TwoAdicFriPcs<Val, Radix2DitParallel, Mmcs, ExtensionMmcs>` of p3-fri 0.5.1
// (rev e9d75614, not vendored) -- as the reference's prover drives it: `commit` (src/prover.rs:350,419,
// src/system.rs:193), `commit_ldes` (src/prover.rs:526), `get_evaluations_on_domain` (src/prover.rs:454-468) and
// `open` (src/prover.rs:580). Semantics as published (SURVEY Appendix A.6):
//   opened value  y = P(z), P interpolated from the first n stored rows (the coset GENERATOR * H_n)
//   reduced opening per LDE height:  ro[x] += alpha^{num_reduced} * (Mred(z) - Mred(x)) / (z - x),
//                                    Mred = sum_c alpha^c column_c,  num_reduced += width, x in bit-reversed order
//   commit phase: rows of 2 extension values (ExtensionMmcs -> 4 base columns); after beta
//                 folded[i] = (lo + hi)/2 + beta/2 * g^{-rev(i)} * (lo - hi), then += beta^2 * next input
// The opened values are computed here by a method DIFFERENT from the device's barycentric sums (inverse coset DFT
// + Horner at z); exact arithmetic makes them equal. The Fiat-Shamir control flow of `open` is the product's
// host/pcs.hpp (shared); the independent check of that flow is the restated verifier in cpu_verify.hpp.
// PARITY UNPINNED against real p3-fri outputs: the reference tree holds no golden FRI data.
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use this file.
#pragma once
#include "../multi_stark_b200/host/prover.hpp"
#include "cpu_eval.hpp"
#include "cpu_mmcs.hpp"
#include <list>
#include <omp.h>

namespace orc {
using namespace msh;

struct CpuPcsData : PcsHandle {
    std::vector<Matrix> ldes;  // bit-reversed row order
    MerkleTree tree;
    size_t num_matrices() const override { return ldes.size(); }
    size_t matrix_height(size_t i) const override { return ldes[i].height(); }
    size_t matrix_width(size_t i) const override { return ldes[i].width; }
    void build_tree() {
        std::vector<MatView> views;
        for (auto& m : ldes) views.push_back(MatView{m.values.data(), m.height(), m.width});
        tree = merkle_commit(views);
    }
};

inline std::shared_ptr<CpuPcsData> cpu_commit_ldes(std::vector<Matrix> ldes, Digest& root) {
    auto pd = std::make_shared<CpuPcsData>();
    pd->ldes = std::move(ldes);
    pd->build_tree();
    root = pd->tree.root();
    return pd;
}
inline std::shared_ptr<CpuPcsData> cpu_commit(const std::vector<const Matrix*>& evals, unsigned log_blowup, Digest& root) {
    std::vector<Matrix> ldes;
    for (auto* m : evals) ldes.push_back(coset_lde_batch_bitrev(*m, log_blowup, Fp(GL_GENERATOR)));
    return cpu_commit_ldes(std::move(ldes), root);
}

inline msh::BatchOpening to_host_opening(const orc::BatchOpening& b) {
    msh::BatchOpening o;
    o.opened_values = b.opened_values;
    o.opening_proof = b.opening_proof;
    return o;
}

class CpuOpenDevice : public OpenDevice {
  public:
    CpuOpenDevice(const std::vector<OpenRound>& rounds, unsigned log_blowup) : rounds_(rounds), log_blowup_(log_blowup) {}

    std::vector<OpenedValuesForRound> evaluate() override {
        opened_.clear();
        for (auto& r : rounds_) {
            auto* pd = dynamic_cast<CpuPcsData*>(r.data);
            if (!pd) throw std::runtime_error("open: prover data does not belong to the CPU backend");
            OpenedValuesForRound round_vals;
            for (size_t m = 0; m < pd->ldes.size(); m++) {
                const Matrix& lde = pd->ldes[m];
                std::vector<std::vector<Fp2>> per_point;
                if (!r.points[m].empty()) {
                    // coefficients of every column from the low coset GENERATOR * H_h (stored bit-reversed)
                    size_t h = lde.height() >> log_blowup_, w = lde.width;
                    unsigned lh = log2_strict(h);
                    Matrix nat(h, w);
                    {
                        const long long hh = (long long)h;
#pragma omp parallel for schedule(static)
                        for (long long i = 0; i < hh; i++) {
                            const Fp* src = lde.row(reverse_bits_len((size_t)i, lh));
                            std::copy(src, src + w, nat.row((size_t)i));
                        }
                    }
                    Matrix coeffs = coset_idft_batch(std::move(nat), Fp(GL_GENERATOR));
                    // Horner in row blocks: block b evaluates sum_j c[j0 + j] z^j for every column at once (row-major reads),
                    // the blocks are combined with z^{j0}. Exact field arithmetic: the same values as one long Horner chain.
                    const size_t n_blocks = std::min<size_t>(h, (size_t)omp_get_max_threads() * 8);
                    const size_t bl = (h + n_blocks - 1) / n_blocks;
                    for (const Fp2& z : r.points[m]) {
                        std::vector<Fp2> part(n_blocks * w, Fp2::zero());
#pragma omp parallel for schedule(static)
                        for (long long b = 0; b < (long long)n_blocks; b++) {
                            const size_t j0 = (size_t)b * bl, j1 = std::min(h, j0 + bl);
                            Fp2* acc = part.data() + (size_t)b * w;
                            for (size_t j = j1; j-- > j0;) {
                                const Fp* row = coeffs.row(j);
                                for (size_t c = 0; c < w; c++) acc[c] = acc[c] * z + row[c];
                            }
                        }
                        std::vector<Fp2> ys(w, Fp2::zero());
                        const Fp2 zb = z.pow(bl);
                        for (size_t b = n_blocks; b-- > 0;)  // Horner over the blocks with z^bl
                            for (size_t c = 0; c < w; c++) ys[c] = ys[c] * zb + part[b * w + c];
                        per_point.push_back(std::move(ys));
                    }
                }
                round_vals.push_back(std::move(per_point));
            }
            opened_.push_back(std::move(round_vals));
        }
        return opened_;
    }

    void reduce(Fp2 alpha, unsigned& log_max_height) override {
        std::vector<std::vector<Fp2>> ro(33);
        size_t num_reduced[33] = {0};
        for (size_t ri = 0; ri < rounds_.size(); ri++) {
            auto* pd = dynamic_cast<CpuPcsData*>(rounds_[ri].data);
            for (size_t m = 0; m < pd->ldes.size(); m++) {
                const Matrix& lde = pd->ldes[m];
                size_t H = lde.height(), w = lde.width;
                unsigned lh = log2_strict(H);
                // p3 creates the height's vector for every matrix of every round, opened or not
                if (ro[lh].empty()) ro[lh].assign(H, Fp2::zero());
                if (rounds_[ri].points[m].empty()) continue;
                std::vector<Fp2> apow(w);
                Fp2 acc = Fp2::one();
                for (size_t c = 0; c < w; c++) { apow[c] = acc; acc *= alpha; }
                std::vector<Fp2> mred(H);
                long long hh = (long long)H;
#pragma omp parallel for schedule(static)
                for (long long i = 0; i < hh; i++) {
                    Fp2 s = Fp2::zero();
                    const Fp* row = lde.row((size_t)i);
                    for (size_t c = 0; c < w; c++) s += apow[c] * row[c];
                    mred[i] = s;
                }
                for (size_t p = 0; p < rounds_[ri].points[m].size(); p++) {
                    Fp2 z = rounds_[ri].points[m][p];
                    Fp2 aoff = alpha.pow(num_reduced[lh]);
                    Fp2 yred = Fp2::zero();
                    for (size_t c = 0; c < w; c++) yred += apow[c] * opened_[ri][m][p][c];
                    const std::vector<Fp2>& inv = inverse_denominators(z, lh);
#pragma omp parallel for schedule(static)
                    for (long long i = 0; i < hh; i++) ro[lh][i] += aoff * (yred - mred[i]) * inv[i];
                    num_reduced[lh] += w;
                }
            }
        }
        inputs_.clear();
        for (int lh = 32; lh >= 0; lh--)
            if (!ro[lh].empty()) inputs_.push_back(std::move(ro[lh]));
        if (inputs_.empty()) throw std::runtime_error("open: nothing to open");
        cur_ = inputs_[0];
        next_input_ = 1;
        log_max_height = log2_strict(cur_.size());
    }

    size_t current_len() override { return cur_.size(); }

    Digest commit_round() override {
        // ExtensionMmcs: rows of 2 extension values flattened to 4 base columns
        auto pd = std::make_shared<CpuPcsData>();
        Matrix m(cur_.size() / 2, 4);
        for (size_t i = 0; i < cur_.size(); i++) { m.values[2 * i] = cur_[i].c[0]; m.values[2 * i + 1] = cur_[i].c[1]; }
        pd->ldes.push_back(std::move(m));
        pd->build_tree();
        layers_.push_back(pd);
        return pd->tree.root();
    }

    void fold(Fp2 beta) override {
        size_t half = cur_.size() / 2;
        unsigned lhalf = log2_strict(half);
        Fp ginv = two_adic_generator(lhalf + 1).inverse();
        Fp2 hb = beta.halve();
        std::vector<Fp2> out(half);
        std::vector<Fp> pw(half);
        long long hh = (long long)half;
        const long long CH = 4096;
        long long nch = (hh + CH - 1) / CH;
#pragma omp parallel for schedule(static)
        for (long long ch = 0; ch < nch; ch++) {
            Fp x = ginv.pow((u64)(ch * CH));
            for (long long k = ch * CH; k < std::min(hh, (ch + 1) * CH); k++) { pw[k] = x; x *= ginv; }
        }
#pragma omp parallel for schedule(static)
        for (long long i = 0; i < hh; i++) {
            Fp2 lo = cur_[2 * i], hi = cur_[2 * i + 1];
            Fp gp = pw[reverse_bits_len((size_t)i, lhalf)];
            out[i] = (lo + hi).halve() + hb * (lo - hi) * gp;
        }
        if (next_input_ < inputs_.size() && inputs_[next_input_].size() == half) {
            Fp2 bsq = beta.square();
            for (size_t i = 0; i < half; i++) out[i] += bsq * inputs_[next_input_][i];
            next_input_++;
        }
        cur_ = std::move(out);
    }

    std::vector<Fp2> read_current() override { return cur_; }

    void open_queries(const std::vector<size_t>& indices, const std::vector<unsigned>& round_shifts, size_t n_layers,
                      std::vector<std::vector<msh::BatchOpening>>& rounds_out, std::vector<std::vector<msh::BatchOpening>>& layers_out) override {
        rounds_out.clear();
        layers_out.clear();
        std::vector<size_t> reduced(indices.size());
        for (size_t r = 0; r < round_shifts.size(); r++) {
            for (size_t q = 0; q < indices.size(); q++) reduced[q] = indices[q] >> round_shifts[r];
            rounds_out.push_back(open_round(r, reduced));
        }
        for (size_t k = 0; k < n_layers; k++) {
            for (size_t q = 0; q < indices.size(); q++) reduced[q] = indices[q] >> (k + 1);
            layers_out.push_back(open_layer(k, reduced));
        }
    }

    // test hook: FRI input k (tallest first)
    const std::vector<std::vector<Fp2>>& inputs() const { return inputs_; }

  private:
    // Mmcs::open_batch of round `r` at every index (already reduced to the round's height)
    std::vector<msh::BatchOpening> open_round(size_t r, const std::vector<size_t>& indices) {
        auto* pd = dynamic_cast<CpuPcsData*>(rounds_[r].data);
        std::vector<msh::BatchOpening> out;
        for (size_t i : indices) out.push_back(to_host_opening(open_batch(pd->tree, i)));
        return out;
    }
    // Mmcs::open_batch of commit-phase layer `k` at every pair index
    std::vector<msh::BatchOpening> open_layer(size_t k, const std::vector<size_t>& pair_indices) {
        std::vector<msh::BatchOpening> out;
        for (size_t i : pair_indices) out.push_back(to_host_opening(open_batch(layers_.at(k)->tree, i)));
        return out;
    }
    // 1 / (z - x), x = GENERATOR * w_H^{rev(i)} (p3 `compute_inverse_denominators`), cached per (z, log H)
    const std::vector<Fp2>& inverse_denominators(const Fp2& z, unsigned lh) {
        for (auto& e : invden_)
            if (e.z == z && e.lh == lh) return e.v;
        size_t H = size_t(1) << lh;
        std::vector<Fp2> den(H), inv(H);
        Fp g = two_adic_generator(lh);
        const size_t CH = 4096;
        long long nch = (long long)((H + CH - 1) / CH);
#pragma omp parallel for schedule(static)
        for (long long ch = 0; ch < nch; ch++) {  // x in natural order, scattered to its bit-reversed slot
            size_t lo = (size_t)ch * CH, n = std::min(CH, H - lo);
            Fp x = Fp(GL_GENERATOR) * g.pow(lo);
            for (size_t k = lo; k < lo + n; k++) { den[reverse_bits_len(k, lh)] = z - x; x *= g; }
        }
#pragma omp parallel for schedule(static)
        for (long long ch = 0; ch < nch; ch++) {
            size_t lo = (size_t)ch * CH, n = std::min(CH, H - lo);
            batch_inverse(den.data() + lo, inv.data() + lo, n);
        }
        invden_.push_back(InvDen{z, lh, std::move(inv)});
        return invden_.back().v;
    }
    struct InvDen {
        Fp2 z;
        unsigned lh;
        std::vector<Fp2> v;
    };
    std::list<InvDen> invden_;
    std::vector<OpenRound> rounds_;
    unsigned log_blowup_;
    std::vector<OpenedValuesForRound> opened_;
    std::vector<std::vector<Fp2>> inputs_;
    size_t next_input_ = 0;
    std::vector<Fp2> cur_;
    std::vector<std::shared_ptr<CpuPcsData>> layers_;
};

// The whole prover on the CPU, stage by stage as src/prover.rs:289-603 performs it.
class CpuBackend : public ProverBackend {
  public:
    explicit CpuBackend(const SystemShape& shape) : shape_(shape) {}

    PcsHandlePtr commit(const std::vector<const Matrix*>& evals, Digest& root) override {
        return cpu_commit(evals, (unsigned)shape_.log_blowup(), root);
    }
    PcsHandlePtr commit_stage1(const std::vector<size_t>& circuits, const std::vector<MatrixView>& traces, Digest& root) override {
        active_ = circuits;
        traces_.clear();
        for (auto& v : traces) traces_.push_back(v.to_matrix());
        std::vector<const Matrix*> ptrs;
        for (auto& m : traces_) ptrs.push_back(&m);
        return cpu_commit(ptrs, (unsigned)shape_.log_blowup(), root);
    }
    Fp2 claims_accumulator(const ClaimsView& claims, Fp2 beta, Fp2 gamma) override {
        // src/prover.rs:381-387 (one inversion per claim; the sum is order-independent in exact arithmetic)
        std::vector<Fp2> msgs(claims.size()), inv(claims.size());
        long long n = (long long)claims.size();
#pragma omp parallel for schedule(static)
        for (long long i = 0; i < n; i++) msgs[i] = beta + fingerprint(gamma, claims.at((size_t)i), claims.len((size_t)i));
        const long long CH = 4096;
        long long nch = (n + CH - 1) / CH;
#pragma omp parallel for schedule(static)
        for (long long ch = 0; ch < nch; ch++) batch_inverse(msgs.data() + ch * CH, inv.data() + ch * CH, (size_t)std::min(CH, n - ch * CH));
        Fp2 acc = Fp2::zero();
        for (auto& v : inv) acc += v;
        return acc;
    }
    PcsHandlePtr commit_stage2(Fp2 beta, Fp2 gamma, Fp2 acc, std::vector<Fp2>& intermediate, Digest& root) override {
        std::vector<LookupValues> lvs;
        for (size_t p = 0; p < active_.size(); p++) lvs.push_back(compute_lookup_values(shape_.circuits[active_[p]], traces_[p]));
        std::vector<const LookupValues*> ptrs;
        for (auto& l : lvs) ptrs.push_back(&l);
        std::vector<Matrix> s2;
        stage_2_traces(ptrs, beta, gamma, acc, s2, intermediate);
        std::vector<const Matrix*> evals;
        for (auto& m : s2) evals.push_back(&m);
        return cpu_commit(evals, (unsigned)shape_.log_blowup(), root);
    }
    PcsHandlePtr commit_quotient(const std::vector<QuotientJob>& jobs, PcsHandle* pre, PcsHandle* s1, PcsHandle* s2, Fp2 alpha,
                                 Digest& root) override {
        auto* h1 = dynamic_cast<CpuPcsData*>(s1);
        auto* h2 = dynamic_cast<CpuPcsData*>(s2);
        auto* hp = pre ? dynamic_cast<CpuPcsData*>(pre) : nullptr;
        std::vector<Matrix> ldes;
        for (auto& j : jobs) {
            const Circuit& c = shape_.circuits[j.circuit];
            unsigned lnq = j.log_degree + j.log_quotient_degree;
            DomainView vp{}, v1{h1->ldes[j.pos].values.data(), c.main_width, lnq}, v2{h2->ldes[j.pos].values.data(), c.stage_2_width, lnq};
            bool has_pre = j.preprocessed_idx >= 0 && hp;
            if (has_pre) vp = DomainView{hp->ldes[j.preprocessed_idx].values.data(), c.preprocessed_width, lnq};
            std::vector<Fp2> q = quotient_values(c, j.publics, j.log_degree, j.log_quotient_degree, has_pre ? &vp : nullptr, v1, v2, alpha);
            Matrix flat(q.size(), 2);
            for (size_t i = 0; i < q.size(); i++) { flat.values[2 * i] = q[i].c[0]; flat.values[2 * i + 1] = q[i].c[1]; }
            Matrix sliced = shifted_quotient_slices(std::move(flat), size_t(1) << j.log_quotient_degree);
            ldes.push_back(lde_from_shifted_coefficients(std::move(sliced), (unsigned)shape_.log_blowup()));
        }
        return cpu_commit_ldes(std::move(ldes), root);
    }
    std::unique_ptr<OpenDevice> open_begin(const std::vector<OpenRound>& rounds) override {
        return std::make_unique<CpuOpenDevice>(rounds, (unsigned)shape_.log_blowup());
    }
    void end_proof() override { traces_.clear(); active_.clear(); }

  private:
    const SystemShape& shape_;
    std::vector<size_t> active_;
    std::vector<Matrix> traces_;
};

}  // namespace orc
