// The PCS seen from the prover driver: commitments are made by a backend (device or CPU), the Fiat-Shamir
// transcript of `Pcs::open` is run here, once, over an `OpenDevice` that does the arithmetic between transcript
// steps. Restates the control flow of p3-fri 0.5.1 `TwoAdicFriPcs::open` and `prover::prove_fri` /
// `commit_phase` / `answer_query` (not vendored in the reference; call site src/prover.rs:580), as described in
// SURVEY Appendix A.6:
//   evaluate -> observe every opened value (round, matrix, point, column) -> sample alpha -> reduced openings
//   -> per FRI round: commit pairs, observe root, grind(commit_pow_bits), sample beta, fold (+ beta^2 * next input)
//   -> final polynomial (bit-reversal undone, inverse DFT, truncated), observe -> grind(query_pow_bits)
//   -> num_queries x { index = sample_bits(log_max_height); input openings per round at index >> (log_max - log_h_round);
//                      per FRI layer k the pair index >> (k + 1) with sibling (index >> k) ^ 1 }
// PARITY UNPINNED against real p3 transcripts; the tests check it end to end with a restated verifier.
#pragma once
#include "proof.hpp"
#include <chrono>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>

namespace msh {

struct PcsHandle {  // Pcs::ProverData
    virtual ~PcsHandle() {}
    virtual size_t num_matrices() const = 0;
    virtual size_t matrix_height(size_t i) const = 0;  // LDE height
    virtual size_t matrix_width(size_t i) const = 0;
    size_t max_height() const {
        size_t h = 0;
        for (size_t i = 0; i < num_matrices(); i++) h = std::max(h, matrix_height(i));
        return h;
    }
};
using PcsHandlePtr = std::shared_ptr<PcsHandle>;

// One opening round: a commitment and, per matrix, the points it is opened at (src/prover.rs:540-579).
struct OpenRound {
    PcsHandle* data;
    std::vector<std::vector<Fp2>> points;  // [matrix][point]
};

// The challenges a proof's transcript produced, in order, for the tests that re-derive them with an independent restatement
// of the challenger (tests/_pyverifier.py): beta, gamma, alpha, zeta (prover.hpp), then alpha_pcs and the FRI betas.
struct TranscriptTrace {
    std::vector<Fp2> challenges;
    std::vector<u64> query_indices;
};

struct OpenDevice {
    virtual ~OpenDevice() {}
    std::vector<Fp2> betas;  // the FRI folding challenges, recorded by commit_phase
    // [round][matrix][point][column]
    virtual std::vector<OpenedValuesForRound> evaluate() = 0;
    virtual void reduce(Fp2 alpha, unsigned& log_max_height) = 0;
    virtual size_t current_len() = 0;
    virtual Digest commit_round() = 0;
    virtual void fold(Fp2 beta) = 0;
    virtual std::vector<Fp2> read_current() = 0;
    // FRI commit phase (p3-fri `commit_phase`): commit pairs -> observe root -> grind -> sample beta -> fold, until the vector
    // is stop_len long. A sharded backend overrides it so that only the FRI owner folds and the other ranks replay the
    // transcript from one broadcast.
    virtual void commit_phase(Challenger& ch, size_t stop_len, size_t pow_bits, FriProof& proof) {
        while (current_len() > stop_len) {
            Digest commit = commit_round();
            ch.observe(commit);
            proof.commit_phase_commits.push_back(commit);
            proof.commit_pow_witnesses.push_back(ch.grind(pow_bits));
            Fp2 beta = ch.sample_ext();
            betas.push_back(beta);
            fold(beta);
        }
    }
    // The whole query phase (Mmcs::open_batch of every round and commit-phase layer): round r is opened at
    // indices[q] >> round_shifts[r], layer k at the pair index indices[q] >> (k + 1) (opened row = 2 extension values).
    // rounds_out[r][q], layers_out[k][q].
    virtual void open_queries(const std::vector<size_t>& indices, const std::vector<unsigned>& round_shifts, size_t n_layers,
                              std::vector<std::vector<BatchOpening>>& rounds_out, std::vector<std::vector<BatchOpening>>& layers_out) = 0;
};

inline unsigned log2_exact(size_t n) { return log2_strict(n); }

// Naive inverse DFT over the extension field (the final polynomial has blowup * final_poly_len points).
inline std::vector<Fp2> idft_ext(const std::vector<Fp2>& evals) {
    size_t n = evals.size();
    unsigned ln = log2_exact(n);
    Fp winv = two_adic_generator(ln).inverse(), ninv = Fp((u64)n).inverse();
    std::vector<Fp2> out(n);
    for (size_t j = 0; j < n; j++) {
        Fp2 acc = Fp2::zero();
        Fp wj = winv.pow((u64)j), cur = Fp::one();
        for (size_t k = 0; k < n; k++) { acc += evals[k] * cur; cur *= wj; }
        out[j] = acc * ninv;
    }
    return out;
}

// TwoAdicFriPcs::open. `rounds_meta[r]` = log2 of the tallest LDE of round r.
inline void pcs_open(OpenDevice& dev, const std::vector<OpenRound>& rounds, const CommitmentParameters& cp, const FriParameters& fp,
                     Challenger& ch, std::vector<OpenedValuesForRound>& opened, FriProof& proof,
                     std::map<std::string, double>* tm = nullptr, TranscriptTrace* trace = nullptr) {
    auto t0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* name) {
        auto t1 = std::chrono::steady_clock::now();
        if (tm) (*tm)[name] += std::chrono::duration<double, std::milli>(t1 - t0).count();
        t0 = t1;
    };
    if (fp.max_log_arity != 1) throw std::runtime_error("only max_log_arity = 1 (binary folding) is supported, as in every reference configuration");
    opened = dev.evaluate();
    for (auto& round : opened)
        for (auto& mat : round)
            for (auto& pt : mat)
                for (auto& y : pt) ch.observe(y);
    lap("fri/evaluate");
    Fp2 alpha = ch.sample_ext();
    unsigned log_max_height = 0;
    dev.reduce(alpha, log_max_height);
    lap("fri/reduce");

    // commit phase
    proof = FriProof();
    const size_t stop_len = (size_t(1) << cp.log_blowup) << fp.log_final_poly_len;
    dev.commit_phase(ch, stop_len, fp.commit_proof_of_work_bits, proof);
    if (trace) {
        trace->challenges.push_back(alpha);
        trace->challenges.insert(trace->challenges.end(), dev.betas.begin(), dev.betas.end());
    }
    lap("fri/commit_phase");
    // final polynomial: undo the bit reversal, inverse DFT, keep final_poly_len coefficients
    std::vector<Fp2> folded = dev.read_current();
    {
        unsigned lf = log2_exact(folded.size());
        std::vector<Fp2> nat(folded.size());
        for (size_t i = 0; i < folded.size(); i++) nat[reverse_bits_len(i, lf)] = folded[i];
        std::vector<Fp2> coeffs = idft_ext(nat);
        size_t keep = size_t(1) << fp.log_final_poly_len;
        for (size_t i = keep; i < coeffs.size(); i++)
            if (!coeffs[i].is_zero()) throw std::runtime_error("FRI final polynomial has degree above the bound (invalid witness?)");
        coeffs.resize(keep);
        proof.final_poly = coeffs;
    }
    for (auto& c : proof.final_poly) ch.observe(c);
    proof.query_pow_witness = ch.grind(fp.query_proof_of_work_bits);

    lap("fri/final_poly");
    // query phase: sample all indices (no observation happens in between), then open in batches
    std::vector<size_t> indices(fp.num_queries);
    for (auto& i : indices) i = ch.sample_bits(log_max_height);
    if (trace) trace->query_indices.assign(indices.begin(), indices.end());
    proof.query_proofs.assign(fp.num_queries, QueryProof());
    std::vector<unsigned> round_shifts;
    for (size_t r = 0; r < rounds.size(); r++) round_shifts.push_back(log_max_height - log2_exact(rounds[r].data->max_height()));
    std::vector<std::vector<BatchOpening>> round_ops, layer_ops;
    dev.open_queries(indices, round_shifts, proof.commit_phase_commits.size(), round_ops, layer_ops);
    for (size_t r = 0; r < rounds.size(); r++)
        for (size_t q = 0; q < indices.size(); q++) proof.query_proofs[q].input_proof.push_back(std::move(round_ops[r][q]));
    for (size_t k = 0; k < proof.commit_phase_commits.size(); k++) {
        for (size_t q = 0; q < indices.size(); q++) {
            size_t index_i = indices[q] >> k, sib = (index_i ^ 1) & 1;
            BatchOpening& bo = layer_ops[k][q];
            const std::vector<Fp>& row = bo.opened_values.at(0);
            CommitPhaseProofStep step;
            step.log_arity = 1;
            step.sibling_values.push_back(Fp2(row[2 * sib], row[2 * sib + 1]));
            step.opening_proof = std::move(bo.opening_proof);
            proof.query_proofs[q].commit_phase_openings.push_back(std::move(step));
        }
    }
    lap("fri/queries");
}

// Standalone `Pcs::open` result as bytes (examples/pcs_example.rs:85-105 prints the sizes of exactly these two objects):
// u64 round count, every round's opened values ([matrix][point][column], length-prefixed), then the FRI proof.
inline std::vector<u8> pcs_open_to_bytes(const std::vector<OpenedValuesForRound>& opened, const FriProof& proof) {
    ByteWriter w;
    w.u64_(opened.size());
    for (auto& r : opened) write_opened_round(w, r);
    write_fri_proof(w, proof);
    return w.out;
}

}  // namespace msh
