// libmshost.so: C entry points of the host-side protocol layer (system assembly, workloads and -- in
// prover.hpp -- the prove() driver over the libmsgpu C ABI). Python (tests, bench.py) binds these with ctypes.
#include "system.hpp"
#include "program.hpp"
#include "system_from_graphs.hpp"
#include "gpu_backend.hpp"
#include "dist_backend.hpp"
#include "rowshard_backend.hpp"
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>

using namespace msh;

struct msh_system {
    SystemShape shape;
    std::vector<std::unique_ptr<GraphDesc>> descs;
};

static thread_local std::string g_err;
static thread_local TranscriptTrace g_trace;  // of the last msh_prove on this thread

extern "C" {

const char* msh_last_error() { return g_err.c_str(); }

msh_system* msh_system_create(const char* kind, uint32_t log_blowup, uint32_t log_final_poly_len, uint32_t max_log_arity,
                              uint32_t num_queries, uint32_t commit_pow_bits, uint32_t query_pow_bits) {
    try {
        CommitmentParameters cp;
        cp.log_blowup = log_blowup;
        FriParameters fp;
        fp.log_final_poly_len = log_final_poly_len;
        fp.max_log_arity = max_log_arity;
        fp.num_queries = num_queries;
        fp.commit_proof_of_work_bits = commit_pow_bits;
        fp.query_proof_of_work_bits = query_pow_bits;
        auto sys = std::make_unique<msh_system>();
        sys->shape = SystemShape::build(cp, fp, named_system_inputs(kind));
        for (auto& c : sys->shape.circuits) {
            auto d = std::make_unique<GraphDesc>();
            d->build(c.graph, c.preprocessed_width, c.main_width, c.stage_2_width);
            sys->descs.push_back(std::move(d));
        }
        return sys.release();
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}
// System::new for circuits the caller compiled itself (src/system.rs:115-203 without the named-benchmark shortcut): one
// msgpu_graph_desc per circuit in canonical order; preprocessed[i] = HOST pointer to pre_heights[i] x descs[i].pre_width values
// or NULL. The descriptors are copied. Everything msh_prove / msh_dist_prover_create accept works on the result.
msh_system* msh_system_create_from_graphs(const msgpu_graph_desc* descs, uint32_t n_circuits, const uint64_t* const* preprocessed,
                                          const uint64_t* pre_heights, uint32_t log_blowup, uint32_t log_final_poly_len,
                                          uint32_t max_log_arity, uint32_t num_queries, uint32_t commit_pow_bits,
                                          uint32_t query_pow_bits) {
    try {
        CommitmentParameters cp;
        cp.log_blowup = log_blowup;
        FriParameters fp;
        fp.log_final_poly_len = log_final_poly_len;
        fp.max_log_arity = max_log_arity;
        fp.num_queries = num_queries;
        fp.commit_proof_of_work_bits = commit_pow_bits;
        fp.query_proof_of_work_bits = query_pow_bits;
        auto sys = std::make_unique<msh_system>();
        sys->shape = system_from_descs(cp, fp, descs, n_circuits, preprocessed, pre_heights);
        for (auto& c : sys->shape.circuits) {
            auto d = std::make_unique<GraphDesc>();
            d->build(c.graph, c.preprocessed_width, c.main_width, c.stage_2_width);
            sys->descs.push_back(std::move(d));
        }
        return sys.release();
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}
void msh_system_free(msh_system* s) { delete s; }
uint32_t msh_system_num_circuits(const msh_system* s) { return (uint32_t)s->shape.circuits.size(); }
// out[12]: main_width, pre_width, pre_height, num_lookups, stage2_width, constraint_count, max_constraint_degree,
//          quotient_degree, n_nodes, n_zeros, lookup_prefix_len, preprocessed_index (or ~0)
void msh_circuit_info(const msh_system* s, uint32_t i, uint64_t* out) {
    const Circuit& c = s->shape.circuits[i];
    out[0] = c.main_width; out[1] = c.preprocessed_width; out[2] = c.preprocessed_height; out[3] = c.num_lookups;
    out[4] = c.stage_2_width; out[5] = c.constraint_count; out[6] = c.max_constraint_degree; out[7] = c.quotient_degree();
    out[8] = c.graph.nodes.size(); out[9] = c.graph.zeros.size(); out[10] = c.graph.lookup_prefix_len;
    out[11] = s->shape.preprocessed_indices[i] < 0 ? ~0ull : (uint64_t)s->shape.preprocessed_indices[i];
}
const msgpu_graph_desc* msh_circuit_graph(const msh_system* s, uint32_t i) { return &s->descs[i]->desc; }
void msh_circuit_preprocessed(const msh_system* s, uint32_t i, uint64_t* out) {
    const Circuit& c = s->shape.circuits[i];
    for (size_t k = 0; k < c.preprocessed.values.size(); k++) out[k] = c.preprocessed.values[k].v;
}

// benches/multi_stark.rs:171-238. add_trace_out: next_pow2(num_adds) x 14; claims_out: num_adds x 4
void msh_u32add_workload(uint64_t num_adds, uint64_t* byte_trace_out, uint64_t* add_trace_out, uint64_t* claims_out) {
    auto w = circuits::u32_add_workload(num_adds);
    for (size_t i = 0; i < 256; i++) byte_trace_out[i] = w.byte_trace.values[i].v;
    for (size_t i = 0; i < w.add_trace.values.size(); i++) add_trace_out[i] = w.add_trace.values[i].v;
    if (claims_out)
        for (size_t i = 0; i < w.claims.size(); i++)
            for (int k = 0; k < 4; k++) claims_out[4 * i + k] = w.claims[i][k].v;
}
// same with other xorshift32 seeds: the K circuits of the "multi:K" system get different additions; the byte multiplicities of
// all of them are summed by the caller
void msh_u32add_workload_seeded(uint64_t num_adds, uint32_t seed_a, uint32_t seed_b, uint64_t* byte_trace_out, uint64_t* add_trace_out,
                                uint64_t* claims_out) {
    auto w = circuits::u32_add_workload(num_adds, seed_a, seed_b);
    for (size_t i = 0; i < 256; i++) byte_trace_out[i] = w.byte_trace.values[i].v;
    for (size_t i = 0; i < w.add_trace.values.size(); i++) add_trace_out[i] = w.add_trace.values[i].v;
    if (claims_out)
        for (size_t i = 0; i < w.claims.size(); i++)
            for (int k = 0; k < 4; k++) claims_out[4 * i + k] = w.claims[i][k].v;
}
void msh_wide_trace(uint64_t row0, uint64_t rows, uint64_t width, uint64_t* out) { circuits::wide_cubic_fill(out, row0, rows, width); }
void msh_fib_trace(uint64_t rows, uint64_t* out) {
    Matrix m = circuits::fib_cubic_trace(rows);
    for (size_t i = 0; i < m.values.size(); i++) out[i] = m.values[i].v;
}

// ---- prove(): System::prove_multiple_claims (src/prover.rs:289-603) over the libmsgpu C ABI -----------------------
struct msh_prover {
    msh_system* sys;
    std::unique_ptr<GpuBackend> backend;
    std::unique_ptr<Prover> prover;
};

// Builds the device programs and commits the preprocessed traces (System::new tail, src/system.rs:180-196).
msh_prover* msh_prover_create(msh_system* s, msgpu_ctx* ctx) {
    try {
        auto p = std::make_unique<msh_prover>();
        p->sys = s;
        p->backend = std::make_unique<GpuBackend>(ctx, s->shape);
        p->prover = std::make_unique<Prover>(s->shape, *p->backend);
        return p.release();
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}
// One proof over several GPUs (dist_backend.hpp): every rank creates the prover with the same `owner` (circuit -> rank) and
// its own context, then calls msh_prove with the traces of the circuits it owns (other traces: NULL pointer, true height).
// `comm` is copied; its callbacks must stay valid for the life of the prover. All ranks get the same proof bytes.
msh_prover* msh_dist_prover_create(msh_system* s, msgpu_ctx* ctx, const msh_comm* comm, const int32_t* owner) {
    try {
        auto p = std::make_unique<msh_prover>();
        p->sys = s;
        std::vector<int> own(owner, owner + s->shape.circuits.size());
        p->backend = std::make_unique<DistGpuBackend>(ctx, s->shape, *comm, own);
        p->prover = std::make_unique<Prover>(s->shape, *p->backend);
        return p.release();
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}
// One proof over the ROW SHARDS of every matrix (rowshard_backend.hpp): every rank creates the prover with its own context and
// calls msh_prove with ALL traces (each rank reads only its row block of the tall ones). `comm` needs the device all-to-all and
// all-gather callbacks. All ranks get the same proof bytes, identical to the single-GPU proof.
msh_prover* msh_rowshard_prover_create(msh_system* s, msgpu_ctx* ctx, const msh_comm* comm) {
    try {
        auto p = std::make_unique<msh_prover>();
        p->sys = s;
        p->backend = std::make_unique<RowShardBackend>(ctx, s->shape, *comm);
        p->prover = std::make_unique<Prover>(s->shape, *p->backend);
        return p.release();
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}
// 1 = a height x width trace is read as natural-order row blocks by the row-sharded prover (RowShardBackend::shardable; the rule
// depends on whether peer memory could be set up), 0 = every rank reads all of it, -1 = not a row-sharded prover
int msh_rowshard_shardable(msh_prover* p, uint64_t height, uint64_t width) {
    auto* be = dynamic_cast<RowShardBackend*>(p->backend.get());
    if (!be) return -1;
    return be->shardable((size_t)height, (size_t)width) ? 1 : 0;
}
int msh_rowshard_peer_memory(msh_prover* p) {
    auto* be = dynamic_cast<RowShardBackend*>(p->backend.get());
    return be && be->peer_memory() ? 1 : 0;
}
uint64_t msh_rowshard_peer_bytes(msh_prover* p) {
    auto* be = dynamic_cast<RowShardBackend*>(p->backend.get());
    return be ? be->peer_bytes() : 0;
}
// Pcs::commit over the row shards alone (bench.py's strong-scaling step): mats[i] = this rank's natural-order ROW BLOCK of matrix
// i (rows [d h / N, (d + 1) h / N) when RowShardProver.shardable(h, w), else the whole matrix), DEVICE pointers (host = 0) or
// HOST pointers to the FULL matrices (host = 1: each rank uploads the rows it reads). Every rank gets the root.
int msh_rowshard_commit(msh_prover* p, const uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths, uint64_t n, int host,
                        uint8_t* root32) {
    try {
        auto* be = dynamic_cast<RowShardBackend*>(p->backend.get());
        if (!be) throw std::runtime_error("not a row-sharded prover");
        std::vector<RowBlocks> blocks;
        for (uint64_t i = 0; i < n; i++) {
            if (host) {
                blocks.push_back(be->upload_blocks(mats[i], (size_t)heights[i], (size_t)widths[i]));
            } else {  // borrowed: the caller's device buffers
                RowBlocks b;
                b.height = (size_t)heights[i];
                b.width = (size_t)widths[i];
                b.whole = !be->shardable(b.height, b.width);
                b.dev = mats[i];
                blocks.push_back(std::move(b));
            }
        }
        Digest root{};
        auto h = be->commit_blocks(blocks, root);
        memcpy(root32, root.data(), 32);
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}
void msh_prover_free(msh_prover* p) { delete p; }
// the preprocessed commitment (verifier key); returns 0 if the system has no preprocessed trace
int msh_prover_preprocessed_commit(const msh_prover* p, uint8_t* out32) {
    const ProverKey& k = p->prover->key();
    if (!k.has_preprocessed) return 0;
    memcpy(out32, k.preprocessed_commit.data(), 32);
    return 1;
}
// traces[i]: HOST heights[i] x main_width of circuit i, canonical values (heights[i] = 0: circuit inactive).
// claims: flat values, offsets[n_claims + 1], or offsets = NULL and claim_stride values per claim. proof_out receives Proof::to_bytes (src/prover.rs:246-249), to be released with
// msh_bytes_free. stage_ms[6] (optional): stage1_commit, claims, stage2_commit, quotient, fri_open, total (host wall clock).
int msh_prove(msh_prover* p, const uint64_t* const* traces, const uint64_t* heights, const uint64_t* claims, const uint64_t* offsets,
              uint64_t claim_stride, uint64_t n_claims, uint8_t** proof_out, uint64_t* proof_len, double* stage_ms) {
    try {
        const SystemShape& shape = p->sys->shape;
        std::vector<MatrixView> views;
        for (size_t i = 0; i < shape.circuits.size(); i++)
            views.push_back(MatrixView((const Fp*)traces[i], (size_t)heights[i], shape.circuits[i].main_width));
        ClaimsView cl;
        cl.values = (const Fp*)claims;
        cl.offsets = offsets;  // NULL: n_claims claims of claim_stride values each
        cl.stride = (size_t)claim_stride;
        cl.n = (size_t)n_claims;
        ProveTimings tm;
        Proof proof = p->prover->prove(cl, views, &tm);
        g_trace = tm.trace;
        std::vector<u8> bytes = proof_to_bytes(proof);
        *proof_out = (uint8_t*)malloc(bytes.size());
        memcpy(*proof_out, bytes.data(), bytes.size());
        *proof_len = bytes.size();
        if (stage_ms) {
            const char* names[5] = {"stark/stage1_commit", "stark/claims", "stark/stage2_commit", "stark/quotient", "stark/fri_open"};
            double total = 0;
            for (int i = 0; i < 5; i++) { stage_ms[i] = tm.ms[names[i]]; total += stage_ms[i]; }
            stage_ms[5] = total;
        }
        if (getenv("MSH_TRACE")) {
            for (auto& kv : tm.ms) fprintf(stderr, "[msh] %-24s %8.3f ms\n", kv.first.c_str(), kv.second);
        }
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}
void msh_bytes_free(uint8_t* b) { free(b); }
// Test hook: the challenges of the last msh_prove on this thread (beta, gamma, alpha, zeta, alpha_pcs, FRI betas; 2 u64 each)
// and its query indices. Returns the number of challenges; writes at most cap of them / cap_idx indices.
uint64_t msh_last_transcript(uint64_t* challenges2, uint64_t cap, uint64_t* indices, uint64_t cap_idx, uint64_t* n_indices) {
    for (size_t i = 0; i < g_trace.challenges.size() && i < cap; i++) {
        challenges2[2 * i] = g_trace.challenges[i].c[0].v;
        challenges2[2 * i + 1] = g_trace.challenges[i].c[1].v;
    }
    for (size_t i = 0; i < g_trace.query_indices.size() && i < cap_idx; i++) indices[i] = g_trace.query_indices[i];
    if (n_indices) *n_indices = g_trace.query_indices.size();
    return g_trace.challenges.size();
}

// ---- standalone PCS use (examples/pcs_example.rs): the transcript object and Pcs::open ------------------------------
struct msh_challenger {
    Challenger ch;
    CommitmentParameters cp;
    FriParameters fp;
};
// GoldilocksBlake3Config::initialise_challenger (src/types.rs:118-130,152-154)
msh_challenger* msh_challenger_create(uint32_t log_blowup, uint32_t log_final_poly_len, uint32_t max_log_arity, uint32_t num_queries,
                                      uint32_t commit_pow_bits, uint32_t query_pow_bits) {
    auto c = std::make_unique<msh_challenger>();
    c->cp.log_blowup = log_blowup;
    c->fp.log_final_poly_len = log_final_poly_len;
    c->fp.max_log_arity = max_log_arity;
    c->fp.num_queries = num_queries;
    c->fp.commit_proof_of_work_bits = commit_pow_bits;
    c->fp.query_proof_of_work_bits = query_pow_bits;
    c->ch = Challenger::for_config(c->cp, c->fp);
    return c.release();
}
void msh_challenger_free(msh_challenger* c) { delete c; }
void msh_challenger_observe_digest(msh_challenger* c, const uint8_t* d32) {
    Digest d;
    memcpy(d.data(), d32, 32);
    c->ch.observe(d);
}
void msh_challenger_observe_values(msh_challenger* c, const uint64_t* v, uint64_t n) {
    for (uint64_t i = 0; i < n; i++) c->ch.observe(Fp(v[i]));
}
void msh_challenger_sample_ext(msh_challenger* c, uint64_t* out2) {
    Fp2 e = c->ch.sample_ext();
    out2[0] = e.c[0].v;
    out2[1] = e.c[1].v;
}

// Pcs::open (call shape of src/prover.rs:580 and examples/pcs_example.rs:85-90): rounds of prover data with, per matrix,
// its opening points (n_points / points as in msgpu_open_begin). out = pcs_open_to_bytes (host/pcs.hpp).
// ms5 (optional): evaluate+begin, reduce, commit phase, final poly, queries.
int msh_pcs_open(msgpu_ctx* ctx, msh_challenger* c, uint64_t n_rounds, msgpu_pdata* const* pds, const uint64_t* n_points,
                 const uint64_t* points, uint8_t** out, uint64_t* out_len, double* ms5) {
    try {
        std::vector<std::unique_ptr<GpuPcsHandle>> handles;
        std::vector<OpenRound> rounds;
        size_t mi = 0, pi = 0;
        for (uint64_t r = 0; r < n_rounds; r++) {
            handles.push_back(std::make_unique<GpuPcsHandle>(pds[r]));  // borrowed
            OpenRound rd;
            rd.data = handles.back().get();
            for (size_t m = 0; m < handles.back()->num_matrices(); m++) {
                std::vector<Fp2> pts;
                for (uint64_t k = 0; k < n_points[mi]; k++, pi++) pts.push_back(Fp2(Fp(points[2 * pi]), Fp(points[2 * pi + 1])));
                mi++;
                rd.points.push_back(std::move(pts));
            }
            rounds.push_back(std::move(rd));
        }
        std::map<std::string, double> tm;
        auto t0 = std::chrono::steady_clock::now();
        GpuOpenDevice dev(ctx, rounds, (uint32_t)c->cp.log_blowup);
        tm["fri/evaluate"] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        std::vector<OpenedValuesForRound> opened;
        FriProof proof;
        pcs_open(dev, rounds, c->cp, c->fp, c->ch, opened, proof, &tm);
        std::vector<u8> bytes = pcs_open_to_bytes(opened, proof);
        *out = (uint8_t*)malloc(bytes.size());
        memcpy(*out, bytes.data(), bytes.size());
        *out_len = bytes.size();
        if (ms5) {
            const char* names[5] = {"fri/evaluate", "fri/reduce", "fri/commit_phase", "fri/final_poly", "fri/queries"};
            for (int i = 0; i < 5; i++) ms5[i] = tm[names[i]];
        }
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}

}  // extern "C"
