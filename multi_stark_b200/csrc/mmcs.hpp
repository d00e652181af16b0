// Device-resident prover data of the mixed-matrix commitment scheme (p3 `MerkleTree` restated for
// the device): matrices in commit order + all digest layers. See merkle.cu for the hash kernels.
#pragma once
#include "internal.hpp"

struct msgpu_pdata {
    struct Mat {
        u64* ptr;
        u64 height, width;
        msg::DevBuf own;  // holds `ptr` when this prover data owns the matrix; empty when it borrows it
        // not empty: `ptr` is still to be written -- the rows are read from these column blocks (pointer, width; dense
        // height x width_b, in column order, possibly in a peer GPU's memory) by the leaf-hash pass, which writes ptr as it goes
        std::vector<std::pair<const u64*, u64>> blocks;
        // a new height x width matrix in an arena block of its own
        static Mat alloc(msg::Ctx& c, u64 height, u64 width) {
            msg::DevBuf b(c, height * width * 8);
            u64* p = b.u();
            return Mat{p, height, width, std::move(b), {}};
        }
    };
    std::vector<Mat> mats;           // original (commit) order
    msg::DevBuf digests;             // all layers back to back
    std::vector<u64> layer_off;      // offset (in digests) of each layer
    std::vector<u64> layer_len;      // layer 0 = leaf digests of the tallest matrices
    u64 max_height = 0;
    u64 total_width = 0;
    uint8_t root[32];
    // Sharded commitments (one proof over several GPUs): a LOCAL part holds this rank's matrices and, per LDE height
    // class, the leaf digests of its rows (no tree: digests == nullptr); the TREE part on the tree owner holds the digest
    // layers built from every rank's class digests (no matrices).
    std::vector<std::pair<u64, msg::DevBuf>> class_leaves;  // (LDE height, 32 * height bytes), tallest first
};

namespace msg {
// Builds the tree over pd->mats (already filled in). Writes pd->root (synchronises the stream).
void mmcs_build(Ctx& c, msgpu_pdata* pd);
// The same without the root read-back: everything is enqueued on the stream, the root is the last digest of pd->digests
// (pd->root is NOT filled in). For the device-side FRI commit phase, which never waits for the host between rounds.
void mmcs_build_async(Ctx& c, msgpu_pdata* pd);
void mmcs_open_batch(Ctx& c, const msgpu_pdata* pd, const u64* indices_host, u64 n_idx, u64* opened_host,
                     uint8_t* proof_host);
// Mmcs::open_batch of several trees in one launch: tree k is opened at indices[q] >> shifts[k]
void mmcs_open_multi(Ctx& c, const msgpu_pdata* const* pds, const u32* shifts, u64 n_trees, const u64* indices_host, u64 n_idx,
                     u64* opened_host, uint8_t* proof_host);
// Local part of a sharded commitment: leaf digests per height class of pd->mats, no node layers.
void mmcs_build_local(Ctx& c, msgpu_pdata* pd);
// Tree part: node layers (with injection) over per-class leaf digests given tallest first; heights strictly decreasing.
void mmcs_build_from_classes(Ctx& c, msgpu_pdata* pd, const std::vector<std::pair<u64, const uint8_t*>>& classes);
// allocates pd->digests for a tree over max_h leaves and fills layer_off / layer_len (layer 0 = leaf digests)
void mmcs_layout_layers(Ctx& c, msgpu_pdata* pd, u64 max_h);
// row block (rows x width) -> column blocks [c0[b], c1[b]), block b a dense rows x (c1[b] - c0[b]) matrix at dst[b] (back to back
// in one buffer, or in the peers' windows); and the inverse, from blocks back to back in src
void pack_column_blocks(Ctx& c, const u64* src, u64 rows, u64 width, const std::vector<u64>& c0, const std::vector<u64>& c1,
                        const std::vector<u64*>& dst);
void interleave_column_blocks(Ctx& c, const u64* src, u64 rows, const std::vector<u64>& widths, u64* dst);
}  // namespace msg
