// BLAKE3 Merkle leaf and node kernels for the mixed-matrix commitment scheme the reference wires at
// src/types.rs:82-84,199-207 (`MerkleTreeMmcs<Val, u8, SerializingHasher<Blake3>,
// CompressionFunctionFromHasher<Blake3, 2, 32>, 2, 32>`):
//   leaf  = BLAKE3(canonical u64 LE bytes of the row; rows of same-height matrices concatenated)
//   node  = BLAKE3(left || right); shorter matrices are injected as H(H(l || r) || leaf(rows_i)).
// Device values are canonical by invariant (gl.cuh), so rows are hashed as stored.
#include "internal.hpp"
#include "blake3.cuh"

namespace msg {

struct LeafMat {
    const u64* ptr;
    u32 width;
    u32 word_off;  // offset of this matrix's words inside the concatenated row message
};
// The matrices of one height class: up to kInlineMats travel as a kernel parameter (no allocation, no upload: a FRI proof
// commits ~20 single-matrix layers), longer lists through device memory.
constexpr int kInlineMats = 8;
struct LeafList {
    LeafMat inl[kInlineMats];
    const LeafMat* ext;
    __device__ __forceinline__ LeafMat at(u32 k) const { return ext ? ext[k] : inl[k]; }
};

// Matrices that are ASSEMBLED while their rows are hashed: the leaf list names the column blocks of such a matrix (dense
// height x width_b each, possibly in another GPU's memory, peer.cu); the staged rows -- all columns, in order -- are also
// written to `dst` (height x width row-major). The row shard of a column-sharded LDE is materialised by the pass that hashes
// it: the blocks are read once (whole lines over NVLink), no separate interleave pass.
constexpr int kMaxAsm = 4;
struct AsmRef {
    u64* dst;
    u32 word_off;  // first word of the matrix inside the concatenated row message
    u32 width;     // columns
};
struct AsmList {
    AsmRef a[kMaxAsm];
    u32 n;
};

constexpr int kLeafThreads = 128;
constexpr int kMaxStack = 24;

// Hash one message of `total_words` 32-bit words provided by get(k).
template <class Get>
__device__ __forceinline__ void hash_words(Get get, u32 total_words, u32 out[8]) {
    const u32 nbytes = total_words * 4u;
    const u32 nchunks = nbytes == 0 ? 1u : (nbytes + 1023u) / 1024u;
    u32 stack[kMaxStack][8];
    u32 sp = 0;
    u32 cv[8];
    for (u32 ci = 0; ci < nchunks; ci++) {
        b3::set_iv(cv);
        const u32 cbytes = min(1024u, nbytes - ci * 1024u);
        const u32 nblocks = cbytes == 0 ? 1u : (cbytes + 63u) / 64u;
        for (u32 b = 0; b < nblocks; b++) {
            u32 m[16];
            const u32 wbase = ci * 256u + b * 16u;
#pragma unroll
            for (int i = 0; i < 16; i++) m[i] = (wbase + i < total_words) ? get(wbase + i) : 0u;
            u32 flags = (b == 0 ? b3::CHUNK_START : 0u) |
                        (b + 1 == nblocks ? (b3::CHUNK_END | (nchunks == 1 ? b3::ROOT : 0u)) : 0u);
            b3::compress(cv, m, ci, 0, min(64u, cbytes - b * 64u), flags);
        }
        if (nchunks == 1) break;
        if (ci + 1 < nchunks) {
            // merge completed subtrees: one parent per trailing zero bit of the chunk count
            u32 total = ci + 1;
            while ((total & 1u) == 0) {
                sp--;
                u32 l[8];
#pragma unroll
                for (int i = 0; i < 8; i++) l[i] = stack[sp][i];
                u32 m[16];
#pragma unroll
                for (int i = 0; i < 8; i++) { m[i] = l[i]; m[8 + i] = cv[i]; }
                b3::set_iv(cv);
                b3::compress(cv, m, 0, 0, 64, b3::PARENT);
                total >>= 1;
            }
#pragma unroll
            for (int i = 0; i < 8; i++) stack[sp][i] = cv[i];
            sp++;
        } else {
            while (sp > 0) {
                sp--;
                u32 m[16];
#pragma unroll
                for (int i = 0; i < 8; i++) { m[i] = stack[sp][i]; m[8 + i] = cv[i]; }
                b3::set_iv(cv);
                b3::compress(cv, m, 0, 0, 64, b3::PARENT | (sp == 0 ? b3::ROOT : 0u));
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = cv[i];
}

// One thread per leaf; rows are staged through shared memory with an odd word pitch so that the
// coalesced global reads turn into conflict-free per-thread row reads.
__global__ void __launch_bounds__(kLeafThreads) k_hash_rows_staged(const __grid_constant__ LeafList mats, u32 nmats, u64 height,
                                                                   u32 total_words, u32 pitch, u32 rows_per_cta,
                                                                   u32* out, const __grid_constant__ AsmList asmb) {
    extern __shared__ u32 sm32[];
    const u64 row0 = (u64)blockIdx.x * rows_per_cta;
    const u32 nrows = (u32)min((u64)rows_per_cta, height - row0);
    for (u32 k = 0; k < nmats; k++) {
        const LeafMat mt = mats.at(k);
        const u64* src = mt.ptr + row0 * mt.width;
        const u32 total = nrows * mt.width;
        for (u32 e = threadIdx.x; e < total; e += blockDim.x) {
            u32 r = e / mt.width, c = e % mt.width;
            u64 v = src[e];
            u32* d = sm32 + (size_t)r * pitch + mt.word_off + 2 * c;
            d[0] = (u32)v;
            d[1] = (u32)(v >> 32);
        }
    }
    __syncthreads();
    // assembled matrices: the staged rows go out as one contiguous run of nrows * width elements (stores are not waited for)
    for (u32 k = 0; k < asmb.n; k++) {
        const AsmRef ar = asmb.a[k];
        u64* dst = ar.dst + row0 * ar.width;
        const u32 total = nrows * ar.width;
        u32 r = threadIdx.x / ar.width, cc = threadIdx.x % ar.width;
        const u32 dr = blockDim.x / ar.width, dc = blockDim.x % ar.width;
        for (u32 e = threadIdx.x; e < total; e += blockDim.x) {
            const u32* s2 = sm32 + (size_t)r * pitch + ar.word_off + 2 * cc;
            dst[e] = (u64)s2[0] | ((u64)s2[1] << 32);
            r += dr;
            cc += dc;
            if (cc >= ar.width) { cc -= ar.width; r++; }
        }
    }
    if (threadIdx.x < nrows) {
        const u32* row = sm32 + (size_t)threadIdx.x * pitch;
        u32 dg[8];
        hash_words([&](u32 k) { return row[k]; }, total_words, dg);
        uint4* o = reinterpret_cast<uint4*>(out + (row0 + threadIdx.x) * 8);
        o[0] = make_uint4(dg[0], dg[1], dg[2], dg[3]);
        o[1] = make_uint4(dg[4], dg[5], dg[6], dg[7]);
    }
}

// Wide rows (more than ~95 columns in total): staging whole rows would leave one warp per CTA hashing (32 rows x 2 KB at 256
// columns), far too few to keep the ALU pipe busy. Here a CTA of 128 threads owns 128 rows and walks the row message in
// segments of kSegWords words (2 BLAKE3 blocks): the segment of all 128 rows is staged with coalesced loads, every thread
// compresses its row's 2 blocks and carries the chunk state (cv, chunk counter, subtree stack) in registers / local memory
// to the next segment. 17 KB of shared memory per CTA: 8 CTAs = 32 hashing warps per SM (64-word segments: 24 warps,
// 6.7 ms instead of 5.4 ms for 2^22 rows of 256 columns; 16-word segments: no further gain).
constexpr int kSegWords = 32;
__global__ void __launch_bounds__(kLeafThreads) k_hash_rows_stream(const __grid_constant__ LeafList mats, u32 nmats, u64 height, u32 total_words,
                                                                   u32* out, const __grid_constant__ AsmList asmb) {
    __shared__ u32 tile[kLeafThreads][kSegWords + 1];
    const u64 row0 = (u64)blockIdx.x * kLeafThreads;
    const u32 nrows = (u32)min((u64)kLeafThreads, height - row0);
    const u32 nbytes = total_words * 4u;
    const u32 nchunks = (nbytes + 1023u) / 1024u;  // >= 2 here
    const bool live = threadIdx.x < nrows;
    u32 stack[kMaxStack][8];
    u32 sp = 0;
    u32 cv[8];
    for (u32 seg0 = 0; seg0 < total_words; seg0 += kSegWords) {
        const u32 seg1 = min(seg0 + (u32)kSegWords, total_words);
        // stage words [seg0, seg1) of every row: per matrix the overlapping columns (word offsets are even: whole u64)
        for (u32 k = 0; k < nmats; k++) {
            const LeafMat mt = mats.at(k);
            const u32 w0 = max(seg0, mt.word_off), w1 = min(seg1, mt.word_off + 2u * mt.width);
            if (w0 >= w1) continue;
            const u32 c0 = (w0 - mt.word_off) >> 1, ncols = (w1 - w0) >> 1, base = w0 - seg0;
            const u64* src = mt.ptr + row0 * mt.width + c0;
            // thread t walks (r, c) pairs t, t + 128, ... with c fastest; the pair is advanced without divisions
            u32 r = threadIdx.x / ncols, cc = threadIdx.x % ncols;
            const u32 dr = kLeafThreads / ncols, dc = kLeafThreads % ncols;
            while (r < nrows) {
                u64 v = src[(u64)r * mt.width + cc];
                tile[r][base + 2 * cc] = (u32)v;
                tile[r][base + 2 * cc + 1] = (u32)(v >> 32);
                r += dr;
                cc += dc;
                if (cc >= ncols) { cc -= ncols; r++; }
            }
        }
        __syncthreads();
        // assembled matrices: the columns of this segment, row by row (up to kSegWords / 2 adjacent elements per row)
        for (u32 k = 0; k < asmb.n; k++) {
            const AsmRef ar = asmb.a[k];
            const u32 w0 = max(seg0, ar.word_off), w1 = min(seg1, ar.word_off + 2u * ar.width);
            if (w0 >= w1) continue;
            const u32 c0 = (w0 - ar.word_off) >> 1, ncols = (w1 - w0) >> 1, base = w0 - seg0;
            u64* dst = ar.dst + row0 * ar.width + c0;
            u32 r = threadIdx.x / ncols, cc = threadIdx.x % ncols;
            const u32 dr = kLeafThreads / ncols, dc = kLeafThreads % ncols;
            while (r < nrows) {
                dst[(u64)r * ar.width + cc] = (u64)tile[r][base + 2 * cc] | ((u64)tile[r][base + 2 * cc + 1] << 32);
                r += dr;
                cc += dc;
                if (cc >= ncols) { cc -= ncols; r++; }
            }
        }
        if (live) {
            const u32* row = tile[threadIdx.x];
#pragma unroll 1
            for (u32 wb = seg0; wb < seg1; wb += 16) {
                const u32 gb = wb >> 4, ci = gb >> 4, bi = gb & 15u;
                const u32 cbytes = min(1024u, nbytes - ci * 1024u);
                const u32 nblocks = (cbytes + 63u) / 64u;
                if (bi == 0) b3::set_iv(cv);
                u32 m[16];
#pragma unroll
                for (int i = 0; i < 16; i++) m[i] = (wb + i < total_words) ? row[wb - seg0 + i] : 0u;
                const u32 flags = (bi == 0 ? b3::CHUNK_START : 0u) | (bi + 1 == nblocks ? b3::CHUNK_END : 0u);
                b3::compress(cv, m, ci, 0, min(64u, cbytes - bi * 64u), flags);
                if (bi + 1 != nblocks) continue;
                // chunk finished: merge completed subtrees (one parent per trailing zero bit of the chunk count), or close the tree
                if (ci + 1 < nchunks) {
                    u32 total = ci + 1;
                    while ((total & 1u) == 0) {
                        sp--;
                        u32 pm[16];
#pragma unroll
                        for (int i = 0; i < 8; i++) { pm[i] = stack[sp][i]; pm[8 + i] = cv[i]; }
                        b3::set_iv(cv);
                        b3::compress(cv, pm, 0, 0, 64, b3::PARENT);
                        total >>= 1;
                    }
#pragma unroll
                    for (int i = 0; i < 8; i++) stack[sp][i] = cv[i];
                    sp++;
                } else {
                    while (sp > 0) {
                        sp--;
                        u32 pm[16];
#pragma unroll
                        for (int i = 0; i < 8; i++) { pm[i] = stack[sp][i]; pm[8 + i] = cv[i]; }
                        b3::set_iv(cv);
                        b3::compress(cv, pm, 0, 0, 64, b3::PARENT | (sp == 0 ? b3::ROOT : 0u));
                    }
                }
            }
        }
        __syncthreads();
    }
    if (live) {
        uint4* o = reinterpret_cast<uint4*>(out + (row0 + threadIdx.x) * 8);
        o[0] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
        o[1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
    }
}

// Fallback for rows too wide to stage (more than ~6000 columns in total): words read from global.
__global__ void __launch_bounds__(kLeafThreads) k_hash_rows_direct(const __grid_constant__ LeafList mats, u32 nmats, u64 height,
                                                                   u32 total_words, u32* out) {
    u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= height) return;
    u32 dg[8];
    hash_words(
        [&](u32 k) {
            u32 mi = 0;
            while (mi + 1 < nmats && mats.at(mi + 1).word_off <= k) mi++;
            const LeafMat mt = mats.at(mi);
            u32 kk = k - mt.word_off;
            u64 v = mt.ptr[r * mt.width + (kk >> 1)];
            return (kk & 1) ? (u32)(v >> 32) : (u32)v;
        },
        total_words, dg);
    uint4* o = reinterpret_cast<uint4*>(out + r * 8);
    o[0] = make_uint4(dg[0], dg[1], dg[2], dg[3]);
    o[1] = make_uint4(dg[4], dg[5], dg[6], dg[7]);
}

// Several node layers per launch: a CTA owns `chunk` adjacent digests of the input layer and reduces them to one,
// level by level through shared memory, writing every intermediate layer to its place in the tree (the prover data
// keeps all layers for the opening proofs). Level l output i = H(in[2i] || in[2i+1]), then H(that || inject_l[i]) when
// matrices of that height are injected.
constexpr int kMaxFusedLevels = 12;
struct SubtreeParams {
    const uint4* in;                        // input layer (global)
    uint4* out[kMaxFusedLevels];            // output layers 1..levels (global, whole-layer base pointers)
    const uint4* inject[kMaxFusedLevels];   // injected leaf digests per output layer or null
    u32 levels;                             // chunk = 1 << levels
};
__device__ __forceinline__ void ld_digest(const uint4* p, u32 d[8]) {
    uint4 a = p[0], b = p[1];
    d[0] = a.x; d[1] = a.y; d[2] = a.z; d[3] = a.w; d[4] = b.x; d[5] = b.y; d[6] = b.z; d[7] = b.w;
}
__device__ __forceinline__ void st_digest(uint4* p, const u32 d[8]) {
    p[0] = make_uint4(d[0], d[1], d[2], d[3]);
    p[1] = make_uint4(d[4], d[5], d[6], d[7]);
}
__global__ void __launch_bounds__(256) k_merkle_subtree(SubtreeParams p) {
    extern __shared__ uint4 sm_t[];
    const u32 chunk = 1u << p.levels;
    uint4* bufA = sm_t;                    // chunk/2 digests
    uint4* bufB = sm_t + chunk;            // chunk/4 digests (2 uint4 per digest)
    const u64 cta = blockIdx.x;
    for (u32 l = 0; l < p.levels; l++) {
        const u32 nodes = chunk >> (l + 1);
        const uint4* src = l == 0 ? p.in + cta * chunk * 2 : ((l & 1) ? bufA : bufB);
        uint4* dst = (l & 1) ? bufB : bufA;
        const u64 gbase = cta * nodes;
        // Levels that keep every thread busy are throughput-bound on the ALU pipe: there the additions go to the FMA pipe as
        // IMAD (blake3.cuh); the upper levels are a latency chain and keep the plain form with the shorter dependency chain.
        const bool wide = nodes >= blockDim.x;
        for (u32 i = threadIdx.x; i < nodes; i += blockDim.x) {
            u32 a[8], b[8], d[8];
            ld_digest(src + 4 * i, a);
            ld_digest(src + 4 * i + 2, b);
            if (wide) b3::hash_pair<true>(a, b, d);
            else b3::hash_pair<false>(a, b, d);
            if (p.inject[l]) {
                u32 x[8], d2[8];
                ld_digest(p.inject[l] + 2 * (gbase + i), x);
                if (wide) b3::hash_pair<true>(d, x, d2);
                else b3::hash_pair<false>(d, x, d2);
#pragma unroll
                for (int k = 0; k < 8; k++) d[k] = d2[k];
            }
            st_digest(dst + 2 * i, d);
            st_digest(p.out[l] + 2 * (gbase + i), d);
        }
        __syncthreads();
    }
}

// raw compression for the known-answer test
__global__ void k_compress_raw(const u32* st, const u32* msg, u32* out) {
    u32 s[16], m[16], o[16];
    for (int i = 0; i < 16; i++) { s[i] = st[i]; m[i] = msg[i]; }
    b3::compress_raw(s, m, o);
    for (int i = 0; i < 16; i++) out[i] = o[i];
}

// ---- BLAKE3 of one long byte string (the transcript's observation buffer) -----------------------------------
// chunk chaining values: one thread per 1024-byte chunk, 16 chained blocks (the last chunk may be short)
__global__ void __launch_bounds__(128) k_b3_chunk_cvs(const uint4* data, u64 len, u64 nchunks, u32* cvs) {
    u64 ci = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (ci >= nchunks) return;
    const u64 cstart = ci * 1024;
    const u32 cbytes = (u32)min((u64)1024, len - cstart);
    const u32 nblocks = cbytes == 0 ? 1u : (cbytes + 63u) / 64u;
    u32 cv[8];
    b3::set_iv(cv);
    const uint8_t* bytes = reinterpret_cast<const uint8_t*>(data);
    for (u32 b = 0; b < nblocks; b++) {
        u32 m[16];
        const u32 blen = min(64u, cbytes - b * 64u);
        if (blen == 64) {
            const uint4* src = data + (cstart + b * 64) / 16;
            uint4 v0 = src[0], v1 = src[1], v2 = src[2], v3 = src[3];
            m[0] = v0.x; m[1] = v0.y; m[2] = v0.z; m[3] = v0.w; m[4] = v1.x; m[5] = v1.y; m[6] = v1.z; m[7] = v1.w;
            m[8] = v2.x; m[9] = v2.y; m[10] = v2.z; m[11] = v2.w; m[12] = v3.x; m[13] = v3.y; m[14] = v3.z; m[15] = v3.w;
        } else {
#pragma unroll
            for (int i = 0; i < 16; i++) {
                u32 w = 0;
                for (int k = 0; k < 4; k++) {
                    u32 off = b * 64u + i * 4u + k;
                    if (off < cbytes) w |= (u32)bytes[cstart + off] << (8 * k);
                }
                m[i] = w;
            }
        }
        u32 flags = (b == 0 ? b3::CHUNK_START : 0u) | (b + 1 == nblocks ? b3::CHUNK_END : 0u);
        b3::compress(cv, m, (u32)ci, (u32)(ci >> 32), blen, flags);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) cvs[ci * 8 + i] = cv[i];
}
// one level of the BLAKE3 tree: adjacent pairs merge, an odd last node moves up unchanged (this reproduces the
// left-heavy tree: the left subtree always holds the largest power of two of chunks)
__global__ void __launch_bounds__(128) k_b3_parent_level(const u32* in, u64 n_in, u32* out) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 n_out = (n_in + 1) / 2;
    if (i >= n_out) return;
    u32 cv[8];
    if (2 * i + 1 < n_in) {
        u32 m[16];
#pragma unroll
        for (int k = 0; k < 16; k++) m[k] = in[(2 * i) * 8 + k];
        b3::set_iv(cv);
        b3::compress(cv, m, 0, 0, 64, b3::PARENT | (n_in == 2 ? b3::ROOT : 0u));
    } else {
#pragma unroll
        for (int k = 0; k < 8; k++) cv[k] = in[(2 * i) * 8 + k];
    }
#pragma unroll
    for (int k = 0; k < 8; k++) out[i * 8 + k] = cv[k];
}

// data_dev: 16-byte aligned device copy of the message (len > 1024). out_dev: 32 bytes.
void b3_hash_long(Ctx& c, const uint8_t* data_dev, u64 len, uint8_t* out_dev) {
    MSG_REQUIRE(len > 1024, "b3_hash_long: message fits one chunk");
    u64 nchunks = (len + 1023) / 1024;
    DevBuf a(c, nchunks * 32), b(c, (nchunks + 1) / 2 * 32);
    launch(c, "k_b3_chunk_cvs", k_b3_chunk_cvs, (unsigned)((nchunks + 127) / 128), 128, 0, (const uint4*)data_dev, len, nchunks, (u32*)a.p);
    u64 n = nchunks;
    while (n > 1) {
        u64 n_out = (n + 1) / 2;
        launch(c, "k_b3_parent_level", k_b3_parent_level, (unsigned)((n_out + 127) / 128), 128, 0, (const u32*)a.p, n, (u32*)b.p);
        std::swap(a, b);
        n = n_out;
    }
    MSG_CUDA(cudaMemcpyAsync(out_dev, a.p, 32, cudaMemcpyDeviceToDevice, c.stream));
}

__global__ void __launch_bounds__(256) k_check_canonical(const u64* v, u64 n, u32* flag) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    bool bad = false;
    for (; i < n; i += (u64)gridDim.x * blockDim.x) bad |= v[i] >= GLD_P;
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1u);
}
// v[i] <- canonical representative (p3's `Goldilocks` may hold any u64 congruent to the value; the device works on canonical ones)
__global__ void __launch_bounds__(256) k_canonicalize(u64* v, u64 n) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i < n; i += (u64)gridDim.x * blockDim.x) {
        u64 x = v[i];
        if (x >= GLD_P) v[i] = x - GLD_P;
    }
}
void canonicalize(Ctx& c, u64* v, u64 n) {
    if (n == 0) return;
    u64 blocks = std::min<u64>((n + 255) / 256, (u64)c.sm_count * 8);
    launch(c, "k_canonicalize", k_canonicalize, (unsigned)std::max<u64>(blocks, 1), 256, 0, v, n);
}
void check_canonical(Ctx& c, const u64* v, u64 n, u32* flag_dev) {
    u64 blocks = std::min<u64>((n + 255) / 256, (u64)c.sm_count * 8);
    launch(c, "k_check_canonical", k_check_canonical, (unsigned)std::max<u64>(blocks, 1), 256, 0, v, n, flag_dev);
}

// dst[r][col0_b + c] = blocks[b][r][c] (the fallback of the assembling leaf kernels)
struct GatherBlocks {
    const u64* blk[16];
    u32 col0[17];
    u32 n;
    u64 rows;
    u64* dst;
};
__global__ void __launch_bounds__(256) k_gather_blocks(const __grid_constant__ GatherBlocks p) {
    const u32 W = p.col0[p.n];
    const u64 total = p.rows * W;
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (u64)gridDim.x * blockDim.x) {
        const u64 r = e / W;
        const u32 col = (u32)(e % W);
        u32 b = 0;
        while (b + 1 < p.n && p.col0[b + 1] <= col) b++;
        p.dst[e] = p.blk[b][r * (p.col0[b + 1] - p.col0[b]) + (col - p.col0[b])];
    }
}

void b3_hash_rows(Ctx& c, const std::vector<MatRef>& mats, uint8_t* digests, const std::vector<AsmTarget>& assemble) {
    MSG_REQUIRE(!mats.empty(), "hash_rows: no matrices");
    u64 height = mats[0].height;
    std::vector<LeafMat> lm;
    std::vector<u32> word_off_of(mats.size(), 0);
    u64 words = 0;
    for (size_t i = 0; i < mats.size(); i++) {
        auto& m = mats[i];
        MSG_REQUIRE(m.height == height, "hash_rows: heights differ");
        MSG_REQUIRE(words + 2 * m.width < (1ull << 30), "hash_rows: row too wide");
        word_off_of[i] = (u32)words;
        if (m.width == 0) continue;
        lm.push_back(LeafMat{m.ptr, (u32)m.width, (u32)words});
        words += 2 * m.width;
    }
    if (height == 0) return;
    // an assembly target that the leaf kernel cannot take (more than kMaxAsm in one class, rows too wide to stage) is gathered by
    // a pass of its own; its blocks are then hashed as they are
    auto gather = [&](const AsmTarget& t) {
        GatherBlocks gb{};
        u64 w = 0;
        for (size_t k = 0; k < t.count; k++) {
            gb.blk[k] = mats[t.first + k].ptr;
            gb.col0[k] = (u32)w;
            w += mats[t.first + k].width;
        }
        gb.col0[t.count] = (u32)w;
        gb.n = (u32)t.count;
        gb.rows = height;
        gb.dst = t.dst;
        if (w == 0) return;
        launch(c, "k_gather_blocks", k_gather_blocks, (unsigned)std::min<u64>((height * w + 255) / 256, (u64)c.sm_count * 16), 256, 0, gb);
    };
    u32 total_words = (u32)words;
    u32 pitch = total_words | 1u;
    size_t budget = 96 * 1024;
    u32 rows = (u32)std::min<size_t>(kLeafThreads, budget / ((size_t)pitch * 4));
    const bool use_stream = rows < (u32)kLeafThreads && total_words * 4u > 1024u && height >= 32;
    const bool use_staged = !use_stream && (rows >= 32 || (u64)rows >= height);
    AsmList asmb{};
    for (auto& t : assemble) {
        MSG_REQUIRE(t.first < mats.size() && t.first + t.count <= mats.size() && t.count >= 1 && t.count <= 16 && t.dst, "hash_rows: bad assembly target");
        u64 w = 0;
        for (size_t k = 0; k < t.count; k++) w += mats[t.first + k].width;
        if (w == 0) continue;
        if (asmb.n < (u32)kMaxAsm && (use_stream || use_staged)) asmb.a[asmb.n++] = AsmRef{t.dst, word_off_of[t.first], (u32)w};
        else gather(t);
    }
    LeafList d_mats{};
    DevBuf d_ext;
    if (lm.size() <= (size_t)kInlineMats) {
        for (size_t k = 0; k < lm.size(); k++) d_mats.inl[k] = lm[k];
    } else {
        d_ext = DevBuf(c, lm.size() * sizeof(LeafMat));
        // the host vector `lm` is copied with a pageable-memory async copy, which is staged before return
        MSG_CUDA(cudaMemcpyAsync(d_ext.p, lm.data(), lm.size() * sizeof(LeafMat), cudaMemcpyHostToDevice, c.stream));
        d_mats.ext = (const LeafMat*)d_ext.p;
    }
    if (use_stream) {
        u64 blocks = (height + kLeafThreads - 1) / kLeafThreads;
        launch(c, "k_hash_rows_stream", k_hash_rows_stream, (unsigned)blocks, kLeafThreads, 0, d_mats, (u32)lm.size(), height, total_words,
               (u32*)digests, asmb);
    } else if (use_staged) {
        if (rows > 32) rows = rows / 32 * 32;
        if (rows == 0) rows = 1;
        ensure_max_smem(k_hash_rows_staged, (int)budget);
        u64 blocks = (height + rows - 1) / rows;
        launch(c, "k_hash_rows_staged", k_hash_rows_staged, (unsigned)blocks, kLeafThreads, (size_t)rows * pitch * 4, d_mats, (u32)lm.size(),
               height, total_words, pitch, rows, (u32*)digests, asmb);
    } else {
        u64 blocks = (height + kLeafThreads - 1) / kLeafThreads;
        launch(c, "k_hash_rows_direct", k_hash_rows_direct, (unsigned)blocks, kLeafThreads, 0, d_mats, (u32)lm.size(), height, total_words,
               (u32*)digests);
    }
}

// Reduces the layer `in` (len digests) by `levels` levels. out[l] / inject[l]: output layer l+1 and its injected digests.
void b3_merkle_subtrees(Ctx& c, const uint8_t* in, u64 len, u32 levels, uint8_t* const* out, const uint8_t* const* inject) {
    MSG_REQUIRE(levels >= 1 && levels <= (u32)kMaxFusedLevels && (len >> levels) >= 1, "merkle: bad fused level count");
    SubtreeParams p{};
    p.in = (const uint4*)in;
    p.levels = levels;
    for (u32 l = 0; l < levels; l++) {
        p.out[l] = (uint4*)out[l];
        p.inject[l] = (const uint4*)inject[l];
    }
    size_t smem = ((size_t)1 << levels) * 24;  // chunk/2 + chunk/4 digests
    ensure_max_smem(k_merkle_subtree, 24 << kMaxFusedLevels);
    u32 threads = (u32)std::min<u64>(256, std::max<u64>(32, (1ull << levels) / 2));
    launch(c, "k_merkle_subtree", k_merkle_subtree, (unsigned)(len >> levels), threads, smem, p);
}

void b3_compress_raw_dev(Ctx& c, const u32* st, const u32* msg, u32* out) {
    launch(c, "k_compress_raw", k_compress_raw, 1, 1, 0, st, msg, out);
}

}  // namespace msg
