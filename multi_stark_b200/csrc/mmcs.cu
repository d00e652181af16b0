// Mixed-matrix Merkle commitment on the device: tree construction with injection of shorter
// matrices and batched query openings. Semantics of p3-merkle-tree `MerkleTreeMmcs::{commit,
// open_batch}` as configured by the reference at src/types.rs:82-84,199-207 (SURVEY Appendix A.4).
#include "mmcs.hpp"
#include <algorithm>
#include <cstring>
#include <numeric>

namespace msg {

struct OpenMat {
    const u64* ptr;
    u32 width;
    u32 shift;    // log_max_height - log_height
    u64 out_off;  // column offset inside one query's opened block
};

// Stable sort of the matrices by height (descending) and the leaf digests of every height class:
// digest[i] = BLAKE3(row i of the class's matrices, concatenated in commit order). `first_out`, when given, receives the
// tallest class (layer 0 of a tree); the other classes get their own buffers. Returns (height, digests), tallest first; the
// first entry's buffer is empty when it went to `first_out`.
static std::vector<std::pair<u64, DevBuf>> hash_classes(Ctx& c, msgpu_pdata* pd, uint8_t* first_out) {
    std::vector<size_t> order(pd->mats.size());
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return pd->mats[a].height > pd->mats[b].height; });
    pd->total_width = 0;
    pd->max_height = 0;
    for (auto& m : pd->mats) {
        MSG_REQUIRE(is_pow2(m.height), "commit: matrix heights must be powers of two");
        pd->total_width += m.width;
        pd->max_height = std::max(pd->max_height, m.height);
    }
    std::vector<std::pair<u64, DevBuf>> classes;
    size_t pos = 0;
    while (pos < order.size()) {
        u64 h = pd->mats[order[pos]].height;
        std::vector<MatRef> group;
        std::vector<AsmTarget> assemble;
        while (pos < order.size() && pd->mats[order[pos]].height == h) {
            auto& m = pd->mats[order[pos++]];
            if (m.blocks.empty()) {
                group.push_back(MatRef{m.ptr, m.height, m.width});
                continue;
            }
            u64 w = 0;
            assemble.push_back(AsmTarget{group.size(), m.blocks.size(), m.ptr});
            for (auto& b : m.blocks) {
                group.push_back(MatRef{b.first, m.height, b.second});
                w += b.second;
            }
            MSG_REQUIRE(w == m.width, "commit: the column blocks of a matrix do not add up to its width");
        }
        DevBuf buf = (classes.empty() && first_out) ? DevBuf() : DevBuf(c, h * 32);
        uint8_t* out = buf ? buf.bytes() : first_out;
        classes.emplace_back(h, std::move(buf));
        b3_hash_rows(c, group, out, assemble);
    }
    for (auto& m : pd->mats) m.blocks.clear();  // every matrix is materialised now
    return classes;
}

void mmcs_layout_layers(Ctx& c, msgpu_pdata* pd, u64 max_h) {
    pd->max_height = max_h;
    pd->digests = DevBuf(c, (2 * max_h - 1) * 32);
    pd->layer_off.clear();
    pd->layer_len.clear();
    u64 off = 0;
    for (u64 len = max_h; len >= 1; len >>= 1) {
        pd->layer_off.push_back(off);
        pd->layer_len.push_back(len);
        off += len;
        if (len == 1) break;
    }
}

// node layers over layer 0 (already in pd->digests) with the shorter classes injected where the layer length equals their
// height: 10 levels per launch while the layer is large, then everything that is left in one CTA
static void build_nodes(Ctx& c, msgpu_pdata* pd, const std::vector<std::pair<u64, const uint8_t*>>& classes) {
    size_t n_layers = pd->layer_len.size();
    std::vector<const uint8_t*> inj(n_layers, nullptr);
    for (size_t k = 1; k < classes.size(); k++) {
        MSG_REQUIRE(classes[k].first < classes[k - 1].first && is_pow2(classes[k].first), "commit: height classes must be distinct powers of two, tallest first");
        inj[ilog2(pd->max_height) - ilog2(classes[k].first)] = classes[k].second;
    }
    size_t l = 0;
    while (l + 1 < n_layers) {
        u64 len = pd->layer_len[l];
        u32 levels = len > 4096 ? 10 : ilog2(len);
        uint8_t* outs[16];
        const uint8_t* injs[16];
        for (u32 k = 0; k < levels; k++) {
            outs[k] = pd->digests.bytes() + pd->layer_off[l + 1 + k] * 32;
            injs[k] = inj[l + 1 + k];
        }
        b3_merkle_subtrees(c, pd->digests.bytes() + pd->layer_off[l] * 32, len, levels, outs, injs);
        l += levels;
    }
}

void mmcs_build(Ctx& c, msgpu_pdata* pd) {
    mmcs_build_async(c, pd);
    MSG_CUDA(cudaMemcpyAsync(pd->root, pd->digests.bytes() + pd->layer_off.back() * 32, 32, cudaMemcpyDeviceToHost, c.stream));
    c.sync();
}

void mmcs_build_async(Ctx& c, msgpu_pdata* pd) {
    StageScope stage_scope(c, "merkle");
    MSG_REQUIRE(!pd->mats.empty(), "commit: no matrices given");
    u64 max_h = 0;
    for (auto& m : pd->mats) max_h = std::max(max_h, m.height);
    MSG_REQUIRE(is_pow2(max_h), "commit: matrix heights must be powers of two");
    mmcs_layout_layers(c, pd, max_h);
    std::vector<std::pair<u64, DevBuf>> cls = hash_classes(c, pd, pd->digests.bytes());
    std::vector<std::pair<u64, const uint8_t*>> view;
    for (auto& cl : cls) view.push_back({cl.first, cl.second ? cl.second.bytes() : pd->digests.bytes()});
    build_nodes(c, pd, view);
}

void mmcs_build_local(Ctx& c, msgpu_pdata* pd) {
    StageScope stage_scope(c, "merkle");
    MSG_REQUIRE(!pd->mats.empty(), "commit: no matrices given");
    pd->class_leaves = hash_classes(c, pd, nullptr);
    pd->layer_off.clear();
    pd->layer_len.clear();
    memset(pd->root, 0, 32);  // rows only: no digest layers
}

void mmcs_build_from_classes(Ctx& c, msgpu_pdata* pd, const std::vector<std::pair<u64, const uint8_t*>>& classes) {
    StageScope stage_scope(c, "merkle");
    MSG_REQUIRE(!classes.empty() && is_pow2(classes[0].first), "tree: no leaf digests given");
    mmcs_layout_layers(c, pd, classes[0].first);
    pd->total_width = 0;
    MSG_CUDA(cudaMemcpyAsync(pd->digests.p, classes[0].second, classes[0].first * 32, cudaMemcpyDeviceToDevice, c.stream));
    build_nodes(c, pd, classes);
    MSG_CUDA(cudaMemcpyAsync(pd->root, pd->digests.bytes() + pd->layer_off.back() * 32, 32, cudaMemcpyDeviceToHost, c.stream));
    c.sync();
}

struct MultiTree {
    const OpenMat* mats;
    const u64* layer_off;
    const uint4* digests;
    u32 nmats, shift, depth, pad;
    u64 tw;           // total width of the tree's matrices
    u64 opened_base;  // u64 offset of this tree's block in the opened output
    u64 proof_base;   // uint4 offset of this tree's block in the proof output
};

__global__ void __launch_bounds__(128) k_open_multi(const MultiTree* trees, const u64* idx, u64* opened, uint4* proofs) {
    const MultiTree t = trees[blockIdx.y];
    const u64 q = blockIdx.x;
    const u64 index = idx[q] >> t.shift;
    u64* o = opened + t.opened_base + q * t.tw;
    for (u32 k = 0; k < t.nmats; k++) {
        const OpenMat m = t.mats[k];
        const u64* row = m.ptr + (index >> m.shift) * m.width;
        for (u32 cidx = threadIdx.x; cidx < m.width; cidx += blockDim.x) o[m.out_off + cidx] = row[cidx];
    }
    uint4* p = proofs + t.proof_base + q * t.depth * 2;
    for (u32 e = threadIdx.x; e < t.depth * 2; e += blockDim.x) {
        u32 lvl = e >> 1, half = e & 1;
        u64 sib = (index >> lvl) ^ 1;
        p[e] = t.digests[(t.layer_off[lvl] + sib) * 2 + half];
    }
}

void mmcs_open_multi(Ctx& c, const msgpu_pdata* const* pds, const u32* shifts, u64 n_trees, const u64* indices_host, u64 n_idx,
                     u64* opened_host, uint8_t* proof_host) {
    if (n_idx == 0 || n_trees == 0) return;
    // one host buffer, one upload: MultiTree[n_trees], the indices, then per tree its OpenMat[] and layer offsets (the
    // descriptors are built here rather than with every tree: a FRI proof commits ~20 layers that are opened once)
    std::vector<MultiTree> mt(n_trees);
    u64 opened_total = 0, proof_total = 0;
    size_t desc_bytes = 0;
    for (u64 k = 0; k < n_trees; k++) {
        const msgpu_pdata* pd = pds[k];
        MSG_REQUIRE(pd && pd->max_height > 0, "open_multi: prover data without a tree");
        for (u64 i = 0; i < n_idx; i++)
            MSG_REQUIRE((indices_host[i] >> shifts[k]) < pd->max_height, "open_multi: index out of range");
        desc_bytes += pd->mats.size() * sizeof(OpenMat) + pd->layer_off.size() * 8;
    }
    const size_t sz_t = n_trees * sizeof(MultiTree), sz_idx = n_idx * 8;
    std::vector<uint8_t> host(sz_t + sz_idx + desc_bytes);
    DevBuf in_buf(c, host.size());
    uint8_t* d_in = in_buf.bytes();
    size_t off = sz_t + sz_idx;
    for (u64 k = 0; k < n_trees; k++) {
        const msgpu_pdata* pd = pds[k];
        u32 depth = pd->digests ? ilog2(pd->max_height) : 0;  // the local part of a sharded commitment has rows only
        MultiTree& t = mt[k];
        t.mats = (const OpenMat*)(d_in + off);
        const u32 log_max = ilog2(pd->max_height);
        u64 col = 0;
        for (auto& m : pd->mats) {
            OpenMat om{m.ptr, (u32)m.width, log_max - ilog2(m.height), col};
            memcpy(host.data() + off, &om, sizeof om);
            off += sizeof om;
            col += m.width;
        }
        t.layer_off = (const u64*)(d_in + off);
        if (!pd->layer_off.empty()) memcpy(host.data() + off, pd->layer_off.data(), pd->layer_off.size() * 8);
        off += pd->layer_off.size() * 8;
        t.digests = (const uint4*)pd->digests.p;
        t.nmats = (u32)pd->mats.size();
        t.shift = shifts[k];
        t.depth = depth;
        t.tw = pd->total_width;
        t.opened_base = opened_total;
        t.proof_base = proof_total * 2;
        opened_total += n_idx * pd->total_width;
        proof_total += n_idx * depth;
    }
    memcpy(host.data(), mt.data(), sz_t);
    memcpy(host.data() + sz_t, indices_host, sz_idx);
    DevBuf d_open(c, std::max<u64>(opened_total * 8, 8)), d_proof(c, std::max<u64>(proof_total * 32, 32));
    MSG_CUDA(cudaMemcpyAsync(d_in, host.data(), host.size(), cudaMemcpyHostToDevice, c.stream));
    launch(c, "k_open_multi", k_open_multi, dim3((unsigned)n_idx, (unsigned)n_trees), 128, 0, (const MultiTree*)d_in, (const u64*)(d_in + sz_t),
           d_open.u(), (uint4*)d_proof.p);
    if (opened_total) MSG_CUDA(cudaMemcpyAsync(opened_host, d_open.p, opened_total * 8, cudaMemcpyDeviceToHost, c.stream));
    if (proof_total) MSG_CUDA(cudaMemcpyAsync(proof_host, d_proof.p, proof_total * 32, cudaMemcpyDeviceToHost, c.stream));
    c.sync();
}

void mmcs_open_batch(Ctx& c, const msgpu_pdata* pd, const u64* indices_host, u64 n_idx, u64* opened_host,
                     uint8_t* proof_host) {
    const u32 shift = 0;
    mmcs_open_multi(c, &pd, &shift, 1, indices_host, n_idx, opened_host, proof_host);
}

// ---- assembling one rank's prover data from a column-block sharded commitment ----------------------------------------
constexpr int kMaxBlocks = 16;
struct InterleaveParams {
    const u64* blocks[kMaxBlocks];
    u32 col0[kMaxBlocks + 1];  // first column of block b; col0[n_blocks] = total width
    u32 n_blocks;
    u64 rows;
    u64* out;
};
// out[r][col0_b + c] = blocks[b][r][c]
__global__ void __launch_bounds__(256) k_interleave_columns(const __grid_constant__ InterleaveParams p) {
    const u32 W = p.col0[p.n_blocks];
    const u64 total = p.rows * W;
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (u64)gridDim.x * blockDim.x) {
        const u64 r = e / W;
        const u32 col = (u32)(e % W);
        u32 b = 0;
        while (b + 1 < p.n_blocks && p.col0[b + 1] <= col) b++;
        const u32 wb = p.col0[b + 1] - p.col0[b];
        p.out[e] = p.blocks[b][r * wb + (col - p.col0[b])];
    }
}

// out[b][r][c] = in[r][col0_b + c]: the inverse (row block -> per-destination column blocks). The row block is read once,
// coalesced; consecutive threads write consecutive addresses of one destination block except at the block boundaries of a row.
struct PackParams {
    const u64* in;
    u64* out[kMaxBlocks];
    u32 col0[kMaxBlocks + 1];
    u32 n_blocks;
    u64 rows;
};
__global__ void __launch_bounds__(256) k_pack_columns(const __grid_constant__ PackParams p) {
    const u32 W = p.col0[p.n_blocks];
    const u64 total = p.rows * W;
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (u64)gridDim.x * blockDim.x) {
        const u64 r = e / W;
        const u32 col = (u32)(e % W);
        u32 b = 0;
        while (b + 1 < p.n_blocks && p.col0[b + 1] <= col) b++;
        const u32 wb = p.col0[b + 1] - p.col0[b];
        p.out[b][r * wb + (col - p.col0[b])] = p.in[e];
    }
}
void pack_column_blocks(Ctx& c, const u64* src, u64 rows, u64 width, const std::vector<u64>& c0, const std::vector<u64>& c1,
                        const std::vector<u64*>& dst) {
    MSG_REQUIRE(!c0.empty() && c0.size() == c1.size() && c0.size() == dst.size() && c0.size() <= (size_t)kMaxBlocks,
                "pack_column_blocks: 1..16 blocks");
    PackParams pp{};
    pp.in = src;
    pp.n_blocks = (u32)c0.size();
    pp.rows = rows;
    for (size_t b = 0; b < c0.size(); b++) {
        MSG_REQUIRE(c0[b] == (b ? c1[b - 1] : 0) && c1[b] >= c0[b], "pack_column_blocks: blocks must tile the columns in order");
        pp.col0[b] = (u32)c0[b];
        pp.out[b] = dst[b];
    }
    MSG_REQUIRE(c1.back() == width, "pack_column_blocks: blocks must cover every column");
    pp.col0[c0.size()] = (u32)width;
    if (rows * width == 0) return;
    launch(c, "k_pack_columns", k_pack_columns, (unsigned)std::min<u64>((rows * width + 255) / 256, (u64)c.sm_count * 16), 256, 0, pp);
}
void interleave_column_blocks(Ctx& c, const u64* src, u64 rows, const std::vector<u64>& widths, u64* dst) {
    MSG_REQUIRE(!widths.empty() && widths.size() <= (size_t)kMaxBlocks, "interleave_column_blocks: 1..16 blocks");
    InterleaveParams ip{};
    ip.n_blocks = (u32)widths.size();
    ip.rows = rows;
    ip.out = dst;
    u64 W = 0;
    for (size_t b = 0; b < widths.size(); b++) {
        ip.blocks[b] = src + rows * W;
        ip.col0[b] = (u32)W;
        W += widths[b];
    }
    ip.col0[widths.size()] = (u32)W;
    if (rows * W == 0) return;
    launch(c, "k_interleave_columns", k_interleave_columns, (unsigned)std::min<u64>((rows * W + 255) / 256, (u64)c.sm_count * 16), 256, 0, ip);
}

}  // namespace msg
