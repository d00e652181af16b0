// ConstraintGraph -> msgpu_graph_desc (the flat arrays the C ABI takes, include/msgpu.h).
#pragma once
#include "expr.hpp"
#include "../../include/msgpu.h"

namespace msh {

struct GraphDesc {
    std::vector<uint8_t> op;
    std::vector<uint32_t> a, b, zeros, lookup_mult, lookup_arg_off, lookup_args;
    std::vector<uint64_t> imm;
    msgpu_graph_desc desc{};

    GraphDesc() = default;
    GraphDesc(const GraphDesc&) = delete;
    GraphDesc& operator=(const GraphDesc&) = delete;

    void build(const ConstraintGraph& g, size_t pre_width, size_t main_width, size_t stage2_width) {
        size_t n = g.nodes.size();
        op.resize(n); a.assign(n, 0); b.assign(n, 0); imm.assign(n, 0);
        for (size_t i = 0; i < n; i++) {
            const Node& nd = g.nodes[i];
            op[i] = (uint8_t)nd.op;
            switch (nd.op) {
                case Op::Const: imm[i] = nd.c.v; break;
                case Op::Var: a[i] = (uint32_t)nd.col.source | ((uint32_t)nd.col.offset << 2); b[i] = nd.col.index; break;
                case Op::Public: a[i] = nd.a; break;
                case Op::Add: case Op::Sub: case Op::Mul: a[i] = nd.a; b[i] = nd.b; break;
                case Op::Neg: a[i] = nd.a; break;
                default: break;
            }
        }
        zeros.assign(g.zeros.begin(), g.zeros.end());
        lookup_mult.clear(); lookup_args.clear(); lookup_arg_off.assign(1, 0);
        for (auto& l : g.lookups) {
            lookup_mult.push_back(l.multiplicity);
            for (u32 x : l.args) lookup_args.push_back(x);
            lookup_arg_off.push_back((uint32_t)lookup_args.size());
        }
        desc.n_nodes = (uint32_t)n;
        desc.op = op.data(); desc.a = a.data(); desc.b = b.data(); desc.imm = imm.data();
        desc.n_zeros = (uint32_t)zeros.size(); desc.zeros = zeros.data();
        desc.n_lookups = (uint32_t)g.lookups.size();
        desc.lookup_mult = lookup_mult.data(); desc.lookup_arg_off = lookup_arg_off.data(); desc.lookup_args = lookup_args.data();
        desc.lookup_prefix_len = (uint32_t)g.lookup_prefix_len;
        desc.pre_width = (uint32_t)pre_width; desc.main_width = (uint32_t)main_width; desc.stage2_width = (uint32_t)stage2_width;
    }
};

// msgpu_graph_desc -> ConstraintGraph: what a caller holding its own compiled circuit (the reference's `ConstraintGraph`,
// src/graph.rs:62-76, produced by its own `compile()`) hands over. Validates what the reference's compiler guarantees
// (children before parents, ids in range) and recomputes the per-node degree multiples (src/graph.rs:240-251).
inline ConstraintGraph graph_from_desc(const msgpu_graph_desc& d) {
    ConstraintGraph g;
    auto fail = [](const std::string& m) { throw std::runtime_error("graph descriptor: " + m); };
    if (d.n_nodes && (!d.op || !d.a || !d.b || !d.imm)) fail("null node arrays");
    for (uint32_t i = 0; i < d.n_nodes; i++) {
        Node n;
        if (d.op[i] > (uint8_t)Op::Neg) fail("unknown op");
        n.op = (Op)d.op[i];
        u32 deg = 0;
        switch (n.op) {
            case Op::Const:
                if (d.imm[i] >= GL_P) fail("constant is not canonical");
                n.c = Fp(d.imm[i]);
                break;
            case Op::Var: {
                uint32_t src = d.a[i] & 3, off = d.a[i] >> 2;
                if (src > 2 || off > 1) fail("bad column reference");
                n.col = ColRef{(Source)src, (RowOffset)off, d.b[i]};
                size_t width = src == 0 ? d.pre_width : src == 1 ? d.main_width : d.stage2_width;
                if (d.b[i] >= width) fail("column index out of range");
                deg = 1;
                break;
            }
            case Op::Public: n.a = d.a[i]; if (n.a >= 8) fail("public index out of range"); break;
            case Op::IsFirstRow: case Op::IsLastRow: deg = 1; break;
            case Op::IsTransition: break;
            case Op::Add: case Op::Sub: case Op::Mul:
                n.a = d.a[i]; n.b = d.b[i];
                if (n.a >= i || n.b >= i) fail("children must precede parents");
                deg = n.op == Op::Mul ? g.degrees[n.a] + g.degrees[n.b] : std::max(g.degrees[n.a], g.degrees[n.b]);
                break;
            case Op::Neg:
                n.a = d.a[i];
                if (n.a >= i) fail("children must precede parents");
                deg = g.degrees[n.a];
                break;
        }
        g.nodes.push_back(n);
        g.degrees.push_back(deg);
    }
    for (uint32_t k = 0; k < d.n_zeros; k++) {
        if (d.zeros[k] >= d.n_nodes) fail("root out of range");
        if (k && d.zeros[k] <= d.zeros[k - 1]) fail("roots must be sorted and distinct (src/graph.rs:155-156)");
        g.zeros.push_back(d.zeros[k]);
        g.max_constraint_degree = std::max(g.max_constraint_degree, g.degrees[d.zeros[k]]);
    }
    if (d.lookup_prefix_len > d.n_nodes) fail("lookup prefix longer than the node vector");
    // lookup values are computed in stage 1, before the stage-2 trace and beta, gamma (publics 0..3) exist (src/graph.rs:343-346)
    for (uint32_t i = 0; i < d.lookup_prefix_len; i++) {
        if (g.nodes[i].op == Op::Public) fail("lookup expression reads a public value");
        if (g.nodes[i].op == Op::Var && g.nodes[i].col.source == Source::Stage2) fail("lookup expression reads a stage-2 column");
    }
    for (uint32_t j = 0; j < d.n_lookups; j++) {
        Lookup<u32> l;
        l.multiplicity = d.lookup_mult[j];
        if (l.multiplicity >= d.lookup_prefix_len) fail("lookup multiplicity outside the lookup prefix");
        for (uint32_t k = d.lookup_arg_off[j]; k < d.lookup_arg_off[j + 1]; k++) {
            if (d.lookup_args[k] >= d.lookup_prefix_len) fail("lookup argument outside the lookup prefix");
            l.args.push_back(d.lookup_args[k]);
        }
        g.lookups.push_back(std::move(l));
    }
    g.lookup_prefix_len = d.lookup_prefix_len;
    return g;
}

}  // namespace msh
