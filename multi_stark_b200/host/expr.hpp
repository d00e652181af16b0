// Frontend expression trees and the constraint compiler: host-side restatement of the reference's
// src/expr.rs (trees with constant folding, :192-244) and src/graph.rs (compile -> flat, hash-consed,
// topologically ordered, base-field-only node vector; :120-188, Interner :215-508). The compiled
// ConstraintGraph is the data format the device quotient / lookup kernels consume (lowered to
// bytecode in program.hpp). Node numbering matters: `zeros` are sorted node ids and that order is the
// alpha-fold order, so interning order follows the reference exactly (lookups first, then base
// constraints, then extension constraints).
#pragma once
#include "goldilocks.hpp"
#include <map>
#include <memory>
#include <stdexcept>
#include <tuple>
#include <vector>
#include <algorithm>

namespace msh {

enum class Source : u8 { Preprocessed = 0, Main = 1, Stage2 = 2 };
enum class RowOffset : u8 { Current = 0, Next = 1 };
struct ColRef {
    Source source;
    RowOffset offset;
    u32 index;
};

enum class Op : u8 { Const = 0, Var = 1, Public = 2, IsFirstRow = 3, IsLastRow = 4, IsTransition = 5, Add = 6, Sub = 7, Mul = 8, Neg = 9 };

// ---- frontend base expression (src/expr.rs:39-51) --------------------------------------------
struct ExprNode;
using ExprPtr = std::shared_ptr<const ExprNode>;
struct ExprNode {
    Op op;
    Fp c;        // Const
    ColRef col;  // Var
    u32 pub;     // Public
    ExprPtr a, b;
};

class Expr {
  public:
    Expr() : p_(mk(Op::Const)) {}
    Expr(Fp c) { auto n = std::make_shared<ExprNode>(); n->op = Op::Const; n->c = c; p_ = n; }
    static Expr constant(Fp c) { return Expr(c); }
    static Expr from_u64(u64 v) { return Expr(Fp(v)); }
    static Expr var(Source s, RowOffset o, u32 index) {
        auto n = std::make_shared<ExprNode>();
        n->op = Op::Var;
        n->col = ColRef{s, o, index};
        return Expr(n);
    }
    static Expr main(u32 i) { return var(Source::Main, RowOffset::Current, i); }
    static Expr main_next(u32 i) { return var(Source::Main, RowOffset::Next, i); }
    static Expr preprocessed(u32 i) { return var(Source::Preprocessed, RowOffset::Current, i); }
    static Expr preprocessed_next(u32 i) { return var(Source::Preprocessed, RowOffset::Next, i); }
    static Expr stage2(u32 i) { return var(Source::Stage2, RowOffset::Current, i); }
    static Expr stage2_next(u32 i) { return var(Source::Stage2, RowOffset::Next, i); }
    static Expr pub(u32 i) { auto n = std::make_shared<ExprNode>(); n->op = Op::Public; n->pub = i; return Expr(n); }
    static Expr is_first_row() { return Expr(mk(Op::IsFirstRow)); }
    static Expr is_last_row() { return Expr(mk(Op::IsLastRow)); }
    static Expr is_transition() { return Expr(mk(Op::IsTransition)); }

    const ExprNode& node() const { return *p_; }
    bool is_const() const { return p_->op == Op::Const; }
    bool is_const(Fp v) const { return is_const() && p_->c == v; }

    // operators fold constants exactly as src/expr.rs:192-244
    friend Expr operator+(const Expr& x, const Expr& y) {
        if (x.is_const() && y.is_const()) return Expr(x.p_->c + y.p_->c);
        if (x.is_const(Fp::zero())) return y;
        if (y.is_const(Fp::zero())) return x;
        return bin(Op::Add, x, y);
    }
    friend Expr operator-(const Expr& x, const Expr& y) {
        if (x.is_const() && y.is_const()) return Expr(x.p_->c - y.p_->c);
        if (y.is_const(Fp::zero())) return x;
        if (x.is_const(Fp::zero())) return -y;
        return bin(Op::Sub, x, y);
    }
    friend Expr operator*(const Expr& x, const Expr& y) {
        if (x.is_const() && y.is_const()) return Expr(x.p_->c * y.p_->c);
        if (x.is_const(Fp::zero()) || y.is_const(Fp::zero())) return Expr(Fp::zero());
        if (x.is_const(Fp::one())) return y;
        if (y.is_const(Fp::one())) return x;
        return bin(Op::Mul, x, y);
    }
    Expr operator-() const {
        if (is_const()) return Expr(-p_->c);
        if (p_->op == Op::Neg) return Expr(p_->a);
        auto n = std::make_shared<ExprNode>();
        n->op = Op::Neg;
        n->a = p_;
        return Expr(n);
    }
    // p3-field `bool_check` = `self.andn(self)` = (ONE - x) * x   (AirBuilder::assert_bool)
    Expr bool_check() const { return (Expr(Fp::one()) - *this) * *this; }

  private:
    explicit Expr(ExprPtr p) : p_(std::move(p)) {}
    static ExprPtr mk(Op op) { auto n = std::make_shared<ExprNode>(); n->op = op; return n; }
    static Expr bin(Op op, const Expr& x, const Expr& y) {
        auto n = std::make_shared<ExprNode>();
        n->op = op;
        n->a = x.p_;
        n->b = y.p_;
        return Expr(n);
    }
    ExprPtr p_;
};

// ---- frontend extension expression (src/expr.rs:56-66); no folding at this level ------------------
struct ExtExprNode;
using ExtExprPtr = std::shared_ptr<const ExtExprNode>;
enum class ExtOp : u8 { Coords, Base, Add, Sub, Mul, Neg };
struct ExtExprNode {
    ExtOp op;
    std::vector<Expr> coords;  // Coords
    Expr base;                 // Base
    ExtExprPtr a, b;
};
class ExtExpr {
  public:
    static ExtExpr coords(std::vector<Expr> c) { auto n = std::make_shared<ExtExprNode>(); n->op = ExtOp::Coords; n->coords = std::move(c); return ExtExpr(n); }
    static ExtExpr from_base(const Expr& e) { auto n = std::make_shared<ExtExprNode>(); n->op = ExtOp::Base; n->base = e; return ExtExpr(n); }
    static ExtExpr constant(const std::vector<Fp>& c) {
        std::vector<Expr> v;
        for (Fp x : c) v.push_back(Expr(x));
        return coords(std::move(v));
    }
    static ExtExpr stage2(u32 slot, u32 d, RowOffset off) {
        std::vector<Expr> v;
        for (u32 j = 0; j < d; j++) v.push_back(Expr::var(Source::Stage2, off, slot * d + j));
        return coords(std::move(v));
    }
    static ExtExpr pub(u32 k, u32 d) {
        std::vector<Expr> v;
        for (u32 j = 0; j < d; j++) v.push_back(Expr::pub(k * d + j));
        return coords(std::move(v));
    }
    friend ExtExpr operator+(const ExtExpr& x, const ExtExpr& y) { return bin(ExtOp::Add, x, y); }
    friend ExtExpr operator-(const ExtExpr& x, const ExtExpr& y) { return bin(ExtOp::Sub, x, y); }
    friend ExtExpr operator*(const ExtExpr& x, const ExtExpr& y) { return bin(ExtOp::Mul, x, y); }
    ExtExpr operator-() const { auto n = std::make_shared<ExtExprNode>(); n->op = ExtOp::Neg; n->a = p_; return ExtExpr(n); }
    const ExtExprNode& node() const { return *p_; }
    bool is_purely_base() const { return purely_base(*p_); }

  private:
    explicit ExtExpr(ExtExprPtr p) : p_(std::move(p)) {}
    static ExtExpr bin(ExtOp op, const ExtExpr& x, const ExtExpr& y) {
        auto n = std::make_shared<ExtExprNode>();
        n->op = op;
        n->a = x.p_;
        n->b = y.p_;
        return ExtExpr(n);
    }
    static bool purely_base(const ExtExprNode& n) {
        switch (n.op) {
            case ExtOp::Coords: return false;
            case ExtOp::Base: return true;
            case ExtOp::Neg: return purely_base(*n.a);
            default: return purely_base(*n.a) && purely_base(*n.b);
        }
    }
    ExtExprPtr p_;
};

// src/lookup.rs:38-75
template <class E>
struct Lookup {
    E multiplicity;
    std::vector<E> args;
    static Lookup push(E m, std::vector<E> a) { return Lookup{std::move(m), std::move(a)}; }
    static Lookup pull(E m, std::vector<E> a) { return Lookup{-m, std::move(a)}; }
};

// src/system.rs:29-35
struct CircuitInputs {
    size_t main_width = 0;
    bool has_preprocessed = false;
    Matrix preprocessed;
    std::vector<Expr> constraints;
    std::vector<ExtExpr> ext_constraints;
    std::vector<Lookup<Expr>> lookups;
};

// src/expr.rs:73-86
struct CircuitSpec {
    size_t main_width = 0, preprocessed_width = 0, stage2_width = 0, num_publics = 0;
    std::vector<Expr> constraints;
    std::vector<ExtExpr> ext_constraints;
    std::vector<Lookup<Expr>> lookups;
};

// ---- compiled graph (src/graph.rs:35-76) ---------------------------------------------------------
struct Node {
    Op op;
    Fp c;         // Const
    ColRef col;   // Var
    u32 a = 0, b = 0;  // children / public index in `a`
};
inline std::tuple<int, u64, int, int, u32, u32, u32> node_key(const Node& n) {
    switch (n.op) {
        case Op::Const: return {(int)n.op, n.c.v, 0, 0, 0, 0, 0};
        case Op::Var: return {(int)n.op, 0, (int)n.col.source, (int)n.col.offset, n.col.index, 0, 0};
        case Op::Public: return {(int)n.op, 0, 0, 0, n.a, 0, 0};
        case Op::IsFirstRow: case Op::IsLastRow: case Op::IsTransition: return {(int)n.op, 0, 0, 0, 0, 0, 0};
        default: return {(int)n.op, 0, 0, 0, 0, n.a, n.b};
    }
}

struct ExtensionParams {
    size_t degree = 2;
    Fp w = Fp(GL_EXT_W);
    bool karatsuba = true;
};

struct ConstraintGraph {
    std::vector<Node> nodes;
    std::vector<u32> degrees;
    std::vector<u32> zeros;
    std::vector<Lookup<u32>> lookups;
    size_t lookup_prefix_len = 0;
    u32 max_constraint_degree = 0;
};

struct CompileError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

class Interner {
  public:
    std::vector<Node> nodes;
    std::vector<u32> degrees;

    u32 intern(const Node& n) {
        auto key = node_key(n);
        auto it = map_.find(key);
        if (it != map_.end()) return it->second;
        u32 id = (u32)nodes.size();
        degrees.push_back(degree_of(n));
        nodes.push_back(n);
        map_[key] = id;
        return id;
    }
    bool as_const(u32 id, Fp* out) const {
        if (nodes[id].op != Op::Const) return false;
        *out = nodes[id].c;
        return true;
    }
    u32 constant(Fp v) { Node n; n.op = Op::Const; n.c = v; return intern(n); }
    u32 add(u32 a, u32 b) {
        Fp x, y;
        bool ca = as_const(a, &x), cb = as_const(b, &y);
        if (ca && cb) return constant(x + y);
        if (ca && !cb && x.is_zero()) return b;
        if (!ca && cb && y.is_zero()) return a;
        if (a > b) std::swap(a, b);
        return intern(binary(Op::Add, a, b));
    }
    u32 sub(u32 a, u32 b) {
        if (a == b) return constant(Fp::zero());
        Fp x, y;
        bool ca = as_const(a, &x), cb = as_const(b, &y);
        if (ca && cb) return constant(x - y);
        if (!ca && cb && y.is_zero()) return a;
        if (ca && !cb && x.is_zero()) return neg(b);
        return intern(binary(Op::Sub, a, b));
    }
    u32 mul(u32 a, u32 b) {
        Fp x, y;
        bool ca = as_const(a, &x), cb = as_const(b, &y);
        if (ca && cb) return constant(x * y);
        if (ca && !cb) {
            if (x.is_zero()) return a;
            if (x == Fp::one()) return b;
        }
        if (!ca && cb) {
            if (y.is_zero()) return b;
            if (y == Fp::one()) return a;
        }
        if (a > b) std::swap(a, b);
        return intern(binary(Op::Mul, a, b));
    }
    u32 neg(u32 a) {
        Fp x;
        if (as_const(a, &x)) return constant(-x);
        if (nodes[a].op == Op::Neg) return nodes[a].a;
        Node n; n.op = Op::Neg; n.a = a;
        return intern(n);
    }

    // allow_public = false: a lookup expression, evaluated in stage 1 before beta and gamma (publics 0..3) are drawn
    u32 compile_expr(const Expr& e, const CircuitSpec& spec, bool allow_stage2, bool allow_public = true) {
        return compile_node(e.node(), spec, allow_stage2, allow_public);
    }

    std::vector<u32> expand_ext(const ExtExpr& e, const CircuitSpec& spec, const ExtensionParams& params, size_t constraint) {
        return expand_node(e.node(), spec, params, constraint);
    }

  private:
    static Node binary(Op op, u32 a, u32 b) { Node n; n.op = op; n.a = a; n.b = b; return n; }
    u32 degree_of(const Node& n) const {
        switch (n.op) {
            case Op::Const: case Op::Public: case Op::IsTransition: return 0;
            case Op::Var: case Op::IsFirstRow: case Op::IsLastRow: return 1;
            case Op::Add: case Op::Sub: return std::max(degrees[n.a], degrees[n.b]);
            case Op::Mul: return degrees[n.a] + degrees[n.b];
            case Op::Neg: return degrees[n.a];
        }
        return 0;
    }
    u32 compile_node(const ExprNode& e, const CircuitSpec& spec, bool allow_stage2, bool allow_public) {
        switch (e.op) {
            case Op::Const: return constant(e.c);
            case Op::Var: {
                size_t width = 0;
                switch (e.col.source) {
                    case Source::Preprocessed: width = spec.preprocessed_width; break;
                    case Source::Main: width = spec.main_width; break;
                    case Source::Stage2:
                        if (!allow_stage2) throw CompileError("Stage2InBaseContext");
                        width = spec.stage2_width;
                        break;
                }
                if (e.col.index >= width) throw CompileError("ColumnOutOfRange");
                Node n; n.op = Op::Var; n.col = e.col;
                return intern(n);
            }
            case Op::Public: {
                if (!allow_public) throw CompileError("PublicInLookup");
                if (e.pub >= spec.num_publics) throw CompileError("PublicOutOfRange");
                Node n; n.op = Op::Public; n.a = e.pub;
                return intern(n);
            }
            case Op::IsFirstRow: case Op::IsLastRow: case Op::IsTransition: { Node n; n.op = e.op; return intern(n); }
            case Op::Add: { u32 a = compile_node(*e.a, spec, allow_stage2, allow_public); u32 b = compile_node(*e.b, spec, allow_stage2, allow_public); return add(a, b); }
            case Op::Sub: { u32 a = compile_node(*e.a, spec, allow_stage2, allow_public); u32 b = compile_node(*e.b, spec, allow_stage2, allow_public); return sub(a, b); }
            case Op::Mul: { u32 a = compile_node(*e.a, spec, allow_stage2, allow_public); u32 b = compile_node(*e.b, spec, allow_stage2, allow_public); return mul(a, b); }
            case Op::Neg: { u32 a = compile_node(*e.a, spec, allow_stage2, allow_public); return neg(a); }
        }
        throw CompileError("bad expression");
    }
    bool is_scalar(const std::vector<u32>& c) const {
        for (size_t i = 1; i < c.size(); i++) {
            Fp v;
            if (!as_const(c[i], &v) || !v.is_zero()) return false;
        }
        return true;
    }
    std::vector<u32> ext_mul(const std::vector<u32>& a, const std::vector<u32>& b, const ExtensionParams& params) {
        size_t d = params.degree;
        std::vector<u32> out;
        if (is_scalar(a)) { for (u32 bk : b) out.push_back(mul(a[0], bk)); return out; }
        if (is_scalar(b)) { for (u32 ak : a) out.push_back(mul(b[0], ak)); return out; }
        if (d == 2 && params.karatsuba) {
            u32 p0 = mul(a[0], b[0]);
            u32 p1 = mul(a[1], b[1]);
            u32 sa = add(a[0], a[1]);
            u32 sb = add(b[0], b[1]);
            u32 s = mul(sa, sb);
            u32 w = constant(params.w);
            u32 wp1 = mul(w, p1);
            u32 c0 = add(p0, wp1);
            u32 t = sub(s, p0);
            u32 c1 = sub(t, p1);
            return {c0, c1};
        }
        u32 w = constant(params.w);
        for (size_t k = 0; k < d; k++) {
            bool hl = false, hh = false;
            u32 low = 0, high = 0;
            for (size_t i = 0; i < d; i++)
                for (size_t j = 0; j < d; j++) {
                    if (i + j == k) { u32 t = mul(a[i], b[j]); low = hl ? add(low, t) : t; hl = true; }
                    else if (i + j == k + d) { u32 t = mul(a[i], b[j]); high = hh ? add(high, t) : t; hh = true; }
                }
            if (hh) { u32 h2 = mul(w, high); out.push_back(add(low, h2)); }
            else out.push_back(low);
        }
        return out;
    }
    std::vector<u32> expand_node(const ExtExprNode& e, const CircuitSpec& spec, const ExtensionParams& params, size_t constraint) {
        size_t d = params.degree;
        switch (e.op) {
            case ExtOp::Coords: {
                if (e.coords.size() != d) throw CompileError("CoordsLength");
                std::vector<u32> out;
                for (auto& c : e.coords) out.push_back(compile_expr(c, spec, true));
                return out;
            }
            case ExtOp::Base: {
                u32 zero = constant(Fp::zero());
                std::vector<u32> out(d, zero);
                out[0] = compile_expr(e.base, spec, true);
                return out;
            }
            case ExtOp::Add: case ExtOp::Sub: {
                auto a = expand_node(*e.a, spec, params, constraint);
                auto b = expand_node(*e.b, spec, params, constraint);
                std::vector<u32> out;
                for (size_t k = 0; k < d; k++) out.push_back(e.op == ExtOp::Add ? add(a[k], b[k]) : sub(a[k], b[k]));
                return out;
            }
            case ExtOp::Neg: {
                auto a = expand_node(*e.a, spec, params, constraint);
                for (auto& c : a) c = neg(c);
                return a;
            }
            case ExtOp::Mul: {
                auto a = expand_node(*e.a, spec, params, constraint);
                auto b = expand_node(*e.b, spec, params, constraint);
                return ext_mul(a, b, params);
            }
        }
        throw CompileError("bad extension expression");
    }
    std::map<std::tuple<int, u64, int, int, u32, u32, u32>, u32> map_;
};

// src/graph.rs:120-188
inline ConstraintGraph compile(const CircuitSpec& spec, const ExtensionParams& params) {
    Interner in;
    ConstraintGraph g;
    for (auto& l : spec.lookups) {
        Lookup<u32> cl;
        cl.multiplicity = in.compile_expr(l.multiplicity, spec, false, false);
        for (auto& a : l.args) cl.args.push_back(in.compile_expr(a, spec, false, false));
        g.lookups.push_back(std::move(cl));
    }
    g.lookup_prefix_len = in.nodes.size();
    auto record_zero = [&](u32 root) {
        Fp c;
        if (in.as_const(root, &c)) {
            if (!c.is_zero()) throw CompileError("UnsatisfiableConstant");
            return;
        }
        g.zeros.push_back(root);
    };
    for (auto& c : spec.constraints) record_zero(in.compile_expr(c, spec, false));
    for (size_t i = 0; i < spec.ext_constraints.size(); i++) {
        if (spec.ext_constraints[i].is_purely_base()) throw CompileError("PurelyBaseExtConstraint");
        for (u32 root : in.expand_ext(spec.ext_constraints[i], spec, params, i)) record_zero(root);
    }
    std::sort(g.zeros.begin(), g.zeros.end());
    g.zeros.erase(std::unique(g.zeros.begin(), g.zeros.end()), g.zeros.end());
    g.max_constraint_degree = 0;
    for (u32 z : g.zeros) g.max_constraint_degree = std::max(g.max_constraint_degree, in.degrees[z]);
    g.nodes = std::move(in.nodes);
    g.degrees = std::move(in.degrees);
    return g;
}

// src/lookup.rs:258-279
inline u32 logup_max_degree(const ConstraintGraph& g) {
    if (g.lookups.empty()) return 1;
    u32 best = 0;
    for (auto& l : g.lookups) {
        u32 md = 0;
        for (u32 a : l.args) md = std::max(md, g.degrees[a]);
        best = std::max(best, std::max(md + 1, g.degrees[l.multiplicity]));
    }
    return best;
}

// src/lookup.rs:325-371 (the executable specification of the logUp constraints; tests only)
inline std::vector<ExtExpr> synthesize_lookups(const std::vector<Lookup<Expr>>& lookups, u32 d) {
    ExtExpr beta = ExtExpr::pub(0, d), gamma = ExtExpr::pub(1, d), acc_initial = ExtExpr::pub(2, d), acc_final = ExtExpr::pub(3, d);
    ExtExpr injection = ExtExpr::from_base(Expr::is_last_row()) * (acc_final - acc_initial);
    if (lookups.empty())
        return {ExtExpr::stage2(0, d, RowOffset::Next) - ExtExpr::stage2(0, d, RowOffset::Current) + injection};
    std::vector<ExtExpr> out;
    size_t last = lookups.size() - 1;
    for (size_t j = 0; j < lookups.size(); j++) {
        ExtExpr source = ExtExpr::stage2((u32)j, d, RowOffset::Current);
        ExtExpr target = j < last ? ExtExpr::stage2((u32)j + 1, d, RowOffset::Current)
                                  : ExtExpr::stage2(0, d, RowOffset::Next) + injection;
        auto& args = lookups[j].args;
        ExtExpr fp = args.empty() ? ExtExpr::from_base(Expr(Fp::zero())) : ExtExpr::from_base(args.back());
        for (size_t i = args.size(); i-- > 1;) fp = fp * gamma + ExtExpr::from_base(args[i - 1]);
        ExtExpr message = beta + fp;
        out.push_back(message * (target - source) - ExtExpr::from_base(lookups[j].multiplicity));
    }
    return out;
}

}  // namespace msh
