// ORACLE C entry points (test infrastructure, not product code). Loaded with ctypes by tests/,
// __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs ONLY.
#include "cpu_dft.hpp"
#include "cpu_mmcs.hpp"
#include <cstring>
#ifdef _OPENMP
#include <omp.h>
#endif

using namespace orc;

static Matrix to_matrix(const u64* in, u64 rows, u64 cols) {
    Matrix m(rows, cols);
    const long long total = (long long)(rows * cols);
#pragma omp parallel for schedule(static)
    for (long long i = 0; i < total; i++) m.values[i] = Fp(in[i]);
    return m;
}
static void from_matrix(const Matrix& m, u64* out) {
    const long long total = (long long)m.values.size();
#pragma omp parallel for schedule(static)
    for (long long i = 0; i < total; i++) out[i] = m.values[i].v;
}

extern "C" {

int orc_num_threads() {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
void orc_set_num_threads(int n) {
#ifdef _OPENMP
    omp_set_num_threads(n);
#else
    (void)n;
#endif
}

// ---- field -------------------------------------------------------------------------------
u64 orc_fp_mul(u64 a, u64 b) { return (Fp(a) * Fp(b)).v; }
u64 orc_fp_inv(u64 a) { return Fp(a).inverse().v; }
u64 orc_two_adic_generator(u32 bits) { return two_adic_generator(bits).v; }
void orc_fp2_mul(const u64* a, const u64* b, u64* out) {
    Fp2 r = Fp2(Fp(a[0]), Fp(a[1])) * Fp2(Fp(b[0]), Fp(b[1]));
    out[0] = r.c[0].v; out[1] = r.c[1].v;
}
void orc_fp2_inv(const u64* a, u64* out) {
    Fp2 r = Fp2(Fp(a[0]), Fp(a[1])).inverse();
    out[0] = r.c[0].v; out[1] = r.c[1].v;
}
// Element-wise host field operations over arrays, for tests/test_host_field.py. Operands of the Fp ops go through Fp(u64),
// so non-canonical inputs are reduced first; the simd:: ops and gl_reduce128 take the raw u64 words.
void orc_fp_op(int op, const u64* a, const u64* b, u64* out, u64 n) {
    for (u64 i = 0; i < n; i++) {
        const Fp x(a[i]), y(b[i]);
        switch (op) {
            case 0: out[i] = x.v; break;
            case 1: out[i] = (x + y).v; break;
            case 2: out[i] = (x - y).v; break;
            case 3: out[i] = (-x).v; break;
            case 4: out[i] = (x * y).v; break;
            case 5: out[i] = x.pow(b[i]).v; break;
            case 6: out[i] = x.inverse().v; break;  // x != 0
            case 7: out[i] = x.halve().v; break;
            case 8: out[i] = simd::gl_mul(a[i], b[i]); break;
            case 9: out[i] = simd::gl_add(a[i], b[i]); break;
            case 10: out[i] = simd::gl_sub(a[i], b[i]); break;
            case 11: out[i] = msh::gl_reduce128(((msh::u128)b[i] << 64) | a[i]); break;  // lo = a, hi = b
            default: out[i] = 0; break;
        }
    }
}
// Fp2 operations over arrays of (c0, c1) pairs: 0 = a * b, 1 = a.inverse() (a != 0), 2 = a.halve()
void orc_fp2_op(int op, const u64* a, const u64* b, u64* out, u64 n) {
    for (u64 i = 0; i < n; i++) {
        const Fp2 x(Fp(a[2 * i]), Fp(a[2 * i + 1])), y(Fp(b[2 * i]), Fp(b[2 * i + 1]));
        const Fp2 r = op == 0 ? x * y : op == 1 ? x.inverse() : x.halve();
        out[2 * i] = r.c[0].v;
        out[2 * i + 1] = r.c[1].v;
    }
}
void orc_fp_batch_inverse(const u64* in, u64* out, u64 n) {
    std::vector<Fp> x(n), r(n);
    for (u64 i = 0; i < n; i++) x[i] = Fp(in[i]);
    batch_inverse(x.data(), r.data(), n);
    for (u64 i = 0; i < n; i++) out[i] = r[i].v;
}
// the oracle's vectorised row kernels (AVX-512 with masked tails, or the auto-vectorised clones under ORC_NO_AVX512)
void orc_dif_butterfly_row(u64* a, u64* b, u64 t, u64 w) { simd::dif_butterfly_row(a, b, t, w); }
void orc_scale_row(u64* dst, const u64* src, u64 s, u64 w) { simd::scale_row(dst, src, s, w); }

// ---- DFT / LDE (p3-dft semantics) ----------------------------------------------------------
void orc_dft_batch(const u64* in, u64 rows, u64 cols, u64* out) { from_matrix(dft_batch(to_matrix(in, rows, cols)), out); }
void orc_dft_batch_bitrev(const u64* in, u64 rows, u64 cols, u64* out) {
    Matrix m = to_matrix(in, rows, cols);
    dft_batch_bitrev_inplace(m.values.data(), rows, cols);
    from_matrix(m, out);
}
void orc_idft_batch(const u64* in, u64 rows, u64 cols, u64* out) { from_matrix(idft_batch(to_matrix(in, rows, cols)), out); }
void orc_coset_dft_batch(const u64* in, u64 rows, u64 cols, u64 shift, u64* out) {
    from_matrix(coset_dft_batch(to_matrix(in, rows, cols), Fp(shift)), out);
}
void orc_coset_idft_batch(const u64* in, u64 rows, u64 cols, u64 shift, u64* out) {
    from_matrix(coset_idft_batch(to_matrix(in, rows, cols), Fp(shift)), out);
}
// out: (rows << added_bits) x cols, bit-reversed storage == what Pcs::commit stores.
void orc_coset_lde_batch_bitrev(const u64* in, u64 rows, u64 cols, u32 added_bits, u64 shift, u64* out) {
    from_matrix(coset_lde_batch_bitrev(to_matrix(in, rows, cols), added_bits, Fp(shift)), out);
}
void orc_lde_from_shifted_coefficients(const u64* in, u64 rows, u64 cols, u32 added_bits, u64* out) {
    from_matrix(lde_from_shifted_coefficients(to_matrix(in, rows, cols), added_bits), out);
}
// shifted_quotient_slices (src/prover.rs:631-679): in = nq x d quotient evaluations (natural order on
// the coset GENERATOR*H_{nq}); out = n x (q*d).
void orc_shifted_quotient_slices(const u64* in, u64 nq, u64 d, u64 q, u64* out) {
    from_matrix(shifted_quotient_slices(to_matrix(in, nq, d), q), out);
}

// ---- hashing / MMCS ------------------------------------------------------------------------
void orc_blake3(const uint8_t* data, u64 len, uint8_t* out32) {
    Digest d = blake3_hash(data, len);
    memcpy(out32, d.data(), 32);
}
void orc_blake3_compress_raw(const u32* state16, const u32* msg16, u32* out16) { b3::compress_raw(state16, msg16, out16); }
void orc_hash_row(const u64* vals, u64 n, uint8_t* out32) {
    std::vector<Fp> v(n);
    for (size_t i = 0; i < n; i++) v[i] = Fp(vals[i]);
    Digest d = hash_values(v.data(), n);
    memcpy(out32, d.data(), 32);
}
void orc_compress(const uint8_t* l, const uint8_t* r, uint8_t* out32) {
    Digest a, b;
    memcpy(a.data(), l, 32); memcpy(b.data(), r, 32);
    Digest d = compress2(a, b);
    memcpy(out32, d.data(), 32);
}

struct OrcTree {
    std::vector<Matrix> mats;
    MerkleTree tree;
};
// Commit to `n` row-major matrices (canonical u64). Returns a handle; root written to root32.
void* orc_mmcs_commit(const u64* const* mats, const u64* heights, const u64* widths, u64 n, uint8_t* root32) {
    auto* t = new OrcTree();
    for (u64 i = 0; i < n; i++) t->mats.push_back(to_matrix(mats[i], heights[i], widths[i]));
    std::vector<MatView> views;
    for (auto& m : t->mats) views.push_back(MatView{m.values.data(), m.height(), m.width});
    try {
        t->tree = merkle_commit(views);
    } catch (const std::exception&) {
        delete t;
        return nullptr;
    }
    memcpy(root32, t->tree.root().data(), 32);
    return t;
}
u64 orc_mmcs_num_layers(void* h) { return ((OrcTree*)h)->tree.digest_layers.size(); }
u64 orc_mmcs_layer_len(void* h, u64 layer) { return ((OrcTree*)h)->tree.digest_layers[layer].size(); }
void orc_mmcs_layer(void* h, u64 layer, uint8_t* out) {
    auto& l = ((OrcTree*)h)->tree.digest_layers[layer];
    for (size_t i = 0; i < l.size(); i++) memcpy(out + 32 * i, l[i].data(), 32);
}
// Opened rows are written back to back (original matrix order); proof = log2(max_height) digests.
void orc_mmcs_open(void* h, u64 index, u64* opened_out, uint8_t* proof_out) {
    BatchOpening bo = open_batch(((OrcTree*)h)->tree, index);
    size_t o = 0;
    for (auto& row : bo.opened_values)
        for (Fp v : row) opened_out[o++] = v.v;
    for (size_t i = 0; i < bo.opening_proof.size(); i++) memcpy(proof_out + 32 * i, bo.opening_proof[i].data(), 32);
}
int orc_mmcs_verify(const uint8_t* root32, const u64* heights, const u64* widths, u64 n, u64 index,
                    const u64* opened, const uint8_t* proof, u64 proof_len) {
    Digest root;
    memcpy(root.data(), root32, 32);
    std::vector<size_t> hs(heights, heights + n);
    std::vector<std::vector<Fp>> ov(n);
    size_t o = 0;
    for (u64 i = 0; i < n; i++)
        for (u64 c = 0; c < widths[i]; c++) ov[i].push_back(Fp(opened[o++]));
    std::vector<Digest> pf(proof_len);
    for (u64 i = 0; i < proof_len; i++) memcpy(pf[i].data(), proof + 32 * i, 32);
    return verify_batch(root, hs, index, ov, pf) ? 1 : 0;
}
void orc_mmcs_free(void* h) { delete (OrcTree*)h; }

}  // extern "C"

// ---- Pcs::commit restated (src/prover.rs:350,419): coset LDE (shift GENERATOR) of every matrix in
// bit-reversed row order, then one MMCS over the LDEs. Returns an OrcTree handle (LDE matrices inside).
extern "C" void* orc_pcs_commit(const u64* const* mats, const u64* heights, const u64* widths, u64 n, u32 log_blowup,
                                uint8_t* root32) {
    auto* t = new OrcTree();
    for (u64 i = 0; i < n; i++)
        t->mats.push_back(coset_lde_batch_bitrev(to_matrix(mats[i], heights[i], widths[i]), log_blowup, Fp(GL_GENERATOR)));
    std::vector<MatView> views;
    for (auto& m : t->mats) views.push_back(MatView{m.values.data(), m.height(), m.width});
    try {
        t->tree = merkle_commit(views);
    } catch (const std::exception&) {
        delete t;
        return nullptr;
    }
    memcpy(root32, t->tree.root().data(), 32);
    return t;
}
extern "C" void orc_mmcs_matrix(void* h, u64 idx, u64* out) { from_matrix(((OrcTree*)h)->mats[idx], out); }
