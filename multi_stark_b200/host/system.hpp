// System assembly on the host: restates src/system.rs (Circuit :52-88, System::new :115-203 without the
// preprocessed commitment, which the prover driver performs through the PCS backend; observe_shape
// :211-222) and the reference's benchmark circuits (benches/multi_stark.rs:73-238).
#pragma once
#include "expr.hpp"
#include "challenger.hpp"

namespace msh {

inline size_t next_pow2(size_t x) {
    size_t p = 1;
    while (p < x) p <<= 1;
    return p;
}

struct Circuit {
    ConstraintGraph graph;
    size_t main_width = 0;
    bool has_preprocessed = false;
    Matrix preprocessed;
    size_t preprocessed_width = 0, preprocessed_height = 0;
    size_t num_lookups = 0;
    size_t stage_2_width = 0;  // max(L,1) * D base columns (src/lookup.rs:90-95)
    size_t num_publics = 0;    // 4 * D
    size_t constraint_count = 0;
    size_t max_constraint_degree = 0;
    // src/system.rs:85-87
    size_t quotient_degree() const { return next_pow2(std::max<size_t>(max_constraint_degree, 2) - 1); }
};

struct SystemShape {
    CommitmentParameters commitment;
    FriParameters fri;
    std::vector<Circuit> circuits;
    std::vector<int> preprocessed_indices;  // position inside the preprocessed commitment, -1 if none
    size_t num_preprocessed = 0;
    size_t log_blowup() const { return commitment.log_blowup; }
    size_t max_quotient_degree() const { return size_t(1) << commitment.log_blowup; }

    static SystemShape build(const CommitmentParameters& cp, const FriParameters& fp, std::vector<CircuitInputs> inputs) {
        SystemShape s;
        s.commitment = cp;
        s.fri = fp;
        ExtensionParams params;
        const size_t d = params.degree;
        for (size_t i = 0; i < inputs.size(); i++) {
            CircuitInputs& in = inputs[i];
            Circuit c;
            c.num_lookups = in.lookups.size();
            c.has_preprocessed = in.has_preprocessed;
            c.preprocessed_width = in.has_preprocessed ? in.preprocessed.width : 0;
            c.preprocessed_height = in.has_preprocessed ? in.preprocessed.height() : 0;
            c.stage_2_width = std::max<size_t>(c.num_lookups, 1) * d;
            c.num_publics = 4 * d;
            CircuitSpec spec;
            spec.main_width = in.main_width;
            spec.preprocessed_width = c.preprocessed_width;
            spec.stage2_width = c.stage_2_width;
            spec.num_publics = c.num_publics;
            spec.constraints = std::move(in.constraints);
            spec.ext_constraints = std::move(in.ext_constraints);
            spec.lookups = std::move(in.lookups);
            c.graph = compile(spec, params);
            c.constraint_count = c.graph.zeros.size() + std::max<size_t>(c.num_lookups, 1) * d;
            c.max_constraint_degree = std::max(c.graph.max_constraint_degree, logup_max_degree(c.graph));
            c.main_width = in.main_width;
            c.preprocessed = std::move(in.preprocessed);
            if (c.quotient_degree() > s.max_quotient_degree())
                throw std::runtime_error("circuit " + std::to_string(i) + ": constraint degree needs a quotient degree the PCS "
                                         "cannot serve; increase log_blowup or lower the constraint degree");
            s.preprocessed_indices.push_back(c.has_preprocessed ? (int)s.num_preprocessed++ : -1);
            s.circuits.push_back(std::move(c));
        }
        return s;
    }

    // The same from circuits that are ALREADY compiled (System::new's per-circuit tail, src/system.rs:146-179, without the
    // compile() call): the caller holds its own ConstraintGraph per circuit.
    struct CompiledInput {
        ConstraintGraph graph;
        size_t main_width = 0;
        bool has_preprocessed = false;
        Matrix preprocessed;
    };
    static SystemShape build_compiled(const CommitmentParameters& cp, const FriParameters& fp, std::vector<CompiledInput> inputs) {
        SystemShape s;
        s.commitment = cp;
        s.fri = fp;
        const size_t d = ExtensionParams().degree;
        for (size_t i = 0; i < inputs.size(); i++) {
            CompiledInput& in = inputs[i];
            Circuit c;
            c.graph = std::move(in.graph);
            c.num_lookups = c.graph.lookups.size();
            c.has_preprocessed = in.has_preprocessed;
            c.preprocessed_width = in.has_preprocessed ? in.preprocessed.width : 0;
            c.preprocessed_height = in.has_preprocessed ? in.preprocessed.height() : 0;
            c.stage_2_width = std::max<size_t>(c.num_lookups, 1) * d;
            c.num_publics = 4 * d;
            c.constraint_count = c.graph.zeros.size() + std::max<size_t>(c.num_lookups, 1) * d;
            c.max_constraint_degree = std::max(c.graph.max_constraint_degree, logup_max_degree(c.graph));
            c.main_width = in.main_width;
            c.preprocessed = std::move(in.preprocessed);
            if (c.quotient_degree() > s.max_quotient_degree())
                throw std::runtime_error("circuit " + std::to_string(i) + ": constraint degree needs a quotient degree the PCS "
                                         "cannot serve; increase log_blowup or lower the constraint degree");
            s.preprocessed_indices.push_back(c.has_preprocessed ? (int)s.num_preprocessed++ : -1);
            s.circuits.push_back(std::move(c));
        }
        return s;
    }

    // src/system.rs:211-222
    void observe_shape(Challenger& ch) const {
        ch.observe_usize(circuits.size());
        for (auto& c : circuits) {
            ch.observe_usize(c.constraint_count);
            ch.observe_usize(c.max_constraint_degree);
            ch.observe_usize(c.preprocessed_height);
            ch.observe_usize(c.preprocessed_width);
            ch.observe_usize(c.main_width);
            ch.observe_usize(c.stage_2_width);
        }
    }
};

// ---- benchmark circuits (benches/multi_stark.rs:73-165) ------------------------------------------
namespace circuits {

inline Expr weighted_u32(u32 c0) {
    return Expr::main(c0) + Expr::main(c0 + 1) * Expr::from_u64(256) + Expr::main(c0 + 2) * Expr::from_u64(256 * 256) +
           Expr::main(c0 + 3) * Expr::from_u64(256 * 256 * 256);
}

// Preprocessed byte table (256 rows, values 0..255); main column = multiplicity.
inline CircuitInputs byte_table() {
    CircuitInputs in;
    in.main_width = 1;
    in.has_preprocessed = true;
    in.preprocessed = Matrix(256, 1);
    for (size_t i = 0; i < 256; i++) in.preprocessed.values[i] = Fp((u64)i);
    in.lookups.push_back(Lookup<Expr>::pull(Expr::main(0), {Expr::from_u64(0), Expr::preprocessed(0)}));
    return in;
}

// U32 addition: x bytes (4) + y bytes (4) + z bytes (4) + carry + multiplicity = 14 columns.
inline CircuitInputs u32_add() {
    CircuitInputs in;
    in.main_width = 14;
    Expr carry = Expr::main(12);
    in.constraints.push_back(carry.bool_check());  // builder.assert_bool(carry)
    // expr1 = x0 + x1*2^8 + x2*2^16 + x3*2^24 + y0 + ...  (left-assoc sums, benches/multi_stark.rs:112-125)
    Expr expr1 = Expr::main(0) + Expr::main(1) * Expr::from_u64(256) + Expr::main(2) * Expr::from_u64(256 * 256) +
                 Expr::main(3) * Expr::from_u64(256 * 256 * 256) + Expr::main(4) + Expr::main(5) * Expr::from_u64(256) +
                 Expr::main(6) * Expr::from_u64(256 * 256) + Expr::main(7) * Expr::from_u64(256 * 256 * 256);
    Expr expr2 = Expr::main(8) + Expr::main(9) * Expr::from_u64(256) + Expr::main(10) * Expr::from_u64(256 * 256) +
                 Expr::main(11) * Expr::from_u64(256 * 256 * 256) + carry * Expr::from_u64(256ull * 256 * 256 * 256);
    in.constraints.push_back(expr1 - expr2);  // builder.assert_eq(expr1, expr2)
    Expr byte_index = Expr::from_u64(0), u32_index = Expr::from_u64(1);
    in.lookups.push_back(Lookup<Expr>::pull(Expr::main(13), {u32_index, weighted_u32(0), weighted_u32(4), weighted_u32(8)}));
    for (u32 i = 0; i < 12; i++) in.lookups.push_back(Lookup<Expr>::push(Expr(Fp::one()), {byte_index, Expr::main(i)}));
    return in;
}

struct U32AddWorkload {
    Matrix byte_trace;  // 256 x 1
    Matrix add_trace;   // next_pow2(num_adds) x 14
    std::vector<std::vector<Fp>> claims;  // [1, x, y, z]
};
// benches/multi_stark.rs:171-238
inline U32AddWorkload u32_add_workload(size_t num_adds, uint32_t seed_a = 0xdeadbeefu, uint32_t seed_b = 0xcafebabeu) {
    U32AddWorkload w;
    size_t h = next_pow2(num_adds);
    w.byte_trace = Matrix(256, 1);
    w.add_trace = Matrix(h, 14);
    w.claims.reserve(num_adds);
    uint32_t a = seed_a, b = seed_b;
    for (size_t r = 0; r < num_adds; r++) {
        a ^= a << 13; a ^= a >> 17; a ^= a << 5;
        b ^= b << 13; b ^= b >> 17; b ^= b << 5;
        uint32_t x = a, y = b, z = x + y;
        uint32_t carry = z < x ? 1 : 0;
        Fp* row = w.add_trace.row(r);
        for (int k = 0; k < 4; k++) {
            uint32_t xb = (x >> (8 * k)) & 0xff, yb = (y >> (8 * k)) & 0xff, zb = (z >> (8 * k)) & 0xff;
            row[k] = Fp(xb); row[4 + k] = Fp(yb); row[8 + k] = Fp(zb);
            w.byte_trace.values[xb] += Fp::one();
            w.byte_trace.values[yb] += Fp::one();
            w.byte_trace.values[zb] += Fp::one();
        }
        row[12] = Fp(carry);
        row[13] = Fp::one();
        w.claims.push_back({Fp(1), Fp(x), Fp(y), Fp(z)});
    }
    return w;
}

}  // namespace circuits
}  // namespace msh

namespace msh {
namespace circuits {

// A lookup-free circuit exercising every selector, next-row reads and a degree-3 constraint (quotient degree 2):
// columns (a, b, c): Fibonacci transition a' = b, b' = a + b from (0, 1), and c = a * b * b on every row.
inline CircuitInputs fib_cubic() {
    CircuitInputs in;
    in.main_width = 3;
    Expr a = Expr::main(0), b = Expr::main(1), c = Expr::main(2);
    in.constraints.push_back(Expr::is_first_row() * a);
    in.constraints.push_back(Expr::is_first_row() * (b - Expr(Fp::one())));
    in.constraints.push_back(Expr::is_transition() * (Expr::main_next(0) - b));
    in.constraints.push_back(Expr::is_transition() * (Expr::main_next(1) - a - b));
    in.constraints.push_back(c - a * b * b);
    in.constraints.push_back(Expr::is_last_row() * Expr::main_next(0));  // the row after the last is row 0, where a = 0
    return in;
}
inline Matrix fib_cubic_trace(size_t rows) {
    Matrix m(rows, 3);
    Fp a = Fp::zero(), b = Fp::one();
    for (size_t r = 0; r < rows; r++) {
        m.row(r)[0] = a; m.row(r)[1] = b; m.row(r)[2] = a * b * b;
        Fp t = a + b; a = b; b = t;
    }
    return m;
}

// BASELINE configs[2]: a wide synthetic AIR without lookups. `width` columns (even); column 2k is free, column 2k+1 is its
// cube: width/2 degree-3 constraints (quotient degree 2, so log_blowup >= 1... the reference needs q <= B).
inline CircuitInputs wide_cubic(size_t width) {
    if (width < 2 || width % 2) throw std::runtime_error("wide circuit needs an even width >= 2");
    CircuitInputs in;
    in.main_width = width;
    for (u32 k = 0; k < width / 2; k++) {
        Expr a = Expr::main(2 * k);
        in.constraints.push_back(Expr::main(2 * k + 1) - a * a * a);
    }
    return in;
}
// counter-based PRNG (splitmix64 of row * width + col) so that any shard of the trace can be generated independently
inline u64 splitmix64(u64 x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
inline void wide_cubic_fill(u64* out, size_t row0, size_t rows, size_t width) {
    for (size_t r = 0; r < rows; r++)
        for (size_t k = 0; k < width / 2; k++) {
            Fp a(splitmix64((u64)(row0 + r) * width + 2 * k) % GL_P);
            out[r * width + 2 * k] = a.v;
            out[r * width + 2 * k + 1] = (a * a * a).v;
        }
}

}  // namespace circuits

// Named systems used by bench.py and the tests (circuit order = matrix order inside every commitment).
//   "u32_add"  : [byte_table, u32_add]                 benches/multi_stark.rs:260-267
//   "mixed"    : [fib_cubic, byte_table, u32_add]      selectors + quotient degree 2 next to the lookup circuits
//   "fib"      : [fib_cubic]
//   "wide:W"   : [wide_cubic(W)]                       BASELINE configs[2] shape (W = 256)
//   "multi:K"  : [byte_table, u32_add x K]             BASELINE configs[3] shape: independent circuits sharing the byte table
inline std::vector<CircuitInputs> named_system_inputs(const std::string& kind) {
    std::vector<CircuitInputs> v;
    if (kind == "u32_add") { v.push_back(circuits::byte_table()); v.push_back(circuits::u32_add()); }
    else if (kind == "mixed") { v.push_back(circuits::fib_cubic()); v.push_back(circuits::byte_table()); v.push_back(circuits::u32_add()); }
    else if (kind == "fib") { v.push_back(circuits::fib_cubic()); }
    else if (kind.rfind("multi:", 0) == 0) {  // BASELINE configs[3] shape: K U32-add circuits (of different heights) + the byte table
        size_t k = (size_t)std::stoul(kind.substr(6));
        if (k < 1 || k > 64) throw std::runtime_error("multi:K needs 1 <= K <= 64");
        v.push_back(circuits::byte_table());
        for (size_t i = 0; i < k; i++) v.push_back(circuits::u32_add());
    }
    else if (kind.rfind("wide:", 0) == 0) { v.push_back(circuits::wide_cubic((size_t)std::stoul(kind.substr(5)))); }
    else throw std::runtime_error("unknown system kind: " + kind);
    return v;
}

}  // namespace msh
