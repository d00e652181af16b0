// Opening phase on the device: barycentric evaluation, reduced openings, FRI fold + commit rounds.
// Restates the arithmetic of p3-fri 0.5.1 `TwoAdicFriPcs::open` / `prove_fri` / `TwoAdicFriFolding::fold_matrix`
// (not vendored in the reference; call site src/prover.rs:580, rounds built at src/prover.rs:540-579); semantics as in
// SURVEY Appendix A.6. PARITY UNPINNED against real p3 outputs (no golden FRI data exists in the reference tree);
// pinned by the tests against the CPU restatement and a restated verifier.
#include "capi_common.hpp"
#include "mmcs.hpp"
#include "blake3.cuh"
#include <algorithm>
#include <cstring>
#include <memory>

namespace msg {

__device__ __forceinline__ u64 fp_inv_d(u64 x) {
    auto sqn = [](u64 v, int n) { for (int i = 0; i < n; i++) v = gl::mul(v, v); return v; };
    u64 t2 = gl::mul(sqn(x, 1), x);
    u64 t4 = gl::mul(sqn(t2, 2), t2);
    u64 t8 = gl::mul(sqn(t4, 4), t4);
    u64 t16 = gl::mul(sqn(t8, 8), t8);
    u64 t24 = gl::mul(sqn(t16, 8), t8);
    u64 t28 = gl::mul(sqn(t24, 4), t4);
    u64 t30 = gl::mul(sqn(t28, 2), t2);
    u64 t31 = gl::mul(sqn(t30, 1), x);
    u64 a = sqn(t31, 1);
    u64 b = gl::mul(a, x);
    return gl::mul(sqn(a, 32), b);
}
__device__ __forceinline__ gl::e2 e2_inverse_d(gl::e2 x) {
    u64 norm = gl::sub(gl::sqr(x.a), gl::mul7(gl::sqr(x.b)));
    u64 ni = fp_inv_d(norm);
    return gl::e2_make(gl::mul(x.a, ni), gl::mul(gl::neg(x.b), ni));
}

// invden[i] = 1 / (z - x_i), x_i = GENERATOR * w_H^{rev(i)}  (the LDE domain in stored order)
constexpr int kInvPerThread = 8;
// Row shards: invden[i] belongs to stored row row0 + i, i < len (unsharded: row0 = 0, len = 2^log_h).
__global__ void __launch_bounds__(256) k_inv_denoms(u64* invden, u32 log_h, gl::e2 z, gl::PowTable xtab, u64 row0, u64 len) {
    const u64 H = len;
    u64 i0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * kInvPerThread;
    if (i0 >= H) return;
    // fully unrolled with constant indices: the batch lives in registers (a dynamically indexed array is local memory)
    const int cnt = (int)min((u64)kInvPerThread, H - i0);
    u64 va[kInvPerThread];
    gl::e2 pref[kInvPerThread];
    gl::e2 acc = gl::e2_make(1, 0);
#pragma unroll
    for (int k = 0; k < kInvPerThread; k++) {
        pref[k] = acc;
        va[k] = 0;
        if (k < cnt) {
            u64 x = gl::pow_lookup(xtab, gl::rev_bits((u32)(row0 + i0 + k), log_h));
            va[k] = gl::sub(z.a, x);
            acc = gl::e2_mul(acc, gl::e2_make(va[k], z.b));
        }
    }
    gl::e2 inv = e2_inverse_d(acc);
#pragma unroll
    for (int k = kInvPerThread - 1; k >= 0; k--) {
        if (k < cnt) {
            gl::e2 r = gl::e2_mul(inv, pref[k]);
            inv = gl::e2_mul(inv, gl::e2_make(va[k], z.b));
            invden[2 * (i0 + k)] = r.a;
            invden[2 * (i0 + k) + 1] = r.b;
        }
    }
}

// Barycentric evaluation on the coset GENERATOR * H_h (the first h stored rows), per column c and point z_p:
//   P_c(z) = (z^h - g^h) / (h g^h) * sum_i M[i][c] * x_i / (z - x_i),   and  x_i / (z - x_i) = z / (z - x_i) - 1,
// so only  S1[c] = sum_i M[i][c]  (base field) and  S2[c][p] = sum_i M[i][c] * invden_p[i]  (extension) are needed:
// the sum is then z * S2 - S1. Terms are accumulated lazily (160-bit, gl::acc_mac) and reduced once per thread.
// partial[cta][c][0] = (S1, 0), partial[cta][c][1 + p] = S2 over the CTA's rows.
constexpr int kMaxPts = 4;
struct BaryParams {
    const u64* M;
    const u64* invden[kMaxPts];
    u64* partial;
    u64 h;
    u32 w, c0, wc;  // this launch covers columns [c0, c0 + wc)
    u32 rows_per_step, tile_rows;
};
// Offset (in u64) of the inverse-denominator tile behind the [tile_rows][wc] matrix tile. It is read and written as
// ulonglong2, so it is rounded up to 16 bytes: tile_rows * wc is odd for some chunk widths (19, 129, ...).
__host__ __device__ __forceinline__ size_t bary_dd_offset(u32 tile_rows, u32 wc) { return ((size_t)tile_rows * wc + 1) & ~(size_t)1; }
// Tiles of tile_rows rows are staged through shared memory with back-to-back coalesced loads (enough bytes in flight to
// keep HBM busy), then thread (column c, row lane) accumulates its rows of the tile.
template <int NPTS>
__global__ void __launch_bounds__(256) k_bary_partial(BaryParams p) {
    extern __shared__ __align__(16) u64 sm_b[];
    const u32 t = threadIdx.x;
    const u32 TR = p.tile_rows, wc = p.wc;
    u64* tile = sm_b;                                                             // [TR][wc]
    ulonglong2* dd = reinterpret_cast<ulonglong2*>(sm_b + bary_dd_offset(TR, wc));  // [TR][NPTS]
    const u32 active = p.rows_per_step * wc;
    const u32 c = t % wc, lane_row = t / wc;
    gl::Acc160 acc[2 * NPTS];
#pragma unroll
    for (int k = 0; k < 2 * NPTS; k++) acc[k] = gl::acc_zero();
    u64 s1 = 0;
    const bool contiguous = (wc == p.w);
    for (u64 row0 = (u64)blockIdx.x * TR; row0 < p.h; row0 += (u64)gridDim.x * TR) {
        const u32 nrows = (u32)min((u64)TR, p.h - row0);
        if (contiguous) {
            const u64* src = p.M + row0 * p.w;
            for (u32 e = t; e < nrows * wc; e += 256) tile[e] = src[e];
        } else {
            for (u32 e = t; e < nrows * wc; e += 256) tile[e] = p.M[(row0 + e / wc) * p.w + p.c0 + e % wc];
        }
        for (u32 e = t; e < nrows * NPTS; e += 256)
            dd[e] = *reinterpret_cast<const ulonglong2*>(p.invden[e % NPTS] + 2 * (row0 + e / NPTS));
        __syncthreads();
        if (t < active) {
            for (u32 r = lane_row; r < nrows; r += p.rows_per_step) {
                const u64 m = tile[r * wc + c];
                s1 = gl::gf::add(s1, m);
#pragma unroll
                for (int k = 0; k < NPTS; k++) {
                    const ulonglong2 d = dd[r * NPTS + k];
                    gl::acc_mac(acc[2 * k], m, d.x);
                    gl::acc_mac(acc[2 * k + 1], m, d.y);
                }
            }
        }
        __syncthreads();
    }
    // reduce over the row lanes of each column (the tile buffer is free again)
    constexpr u32 nslots = NPTS + 1;
    u64* sm = sm_b;  // [rows_per_step][wc][nslots][2]
    if (t < active) {
        u64* o = sm + ((size_t)(lane_row * wc + c) * nslots) * 2;
        o[0] = s1;
        o[1] = 0;
#pragma unroll
        for (int k = 0; k < NPTS; k++) {
            o[2 * (k + 1)] = gl::acc_reduce(acc[2 * k]);
            o[2 * (k + 1) + 1] = gl::acc_reduce(acc[2 * k + 1]);
        }
    }
    __syncthreads();
    if (t < wc) {
        for (u32 k = 0; k < nslots; k++) {
            gl::e2 s = gl::e2_make(0, 0);
            for (u32 l = 0; l < p.rows_per_step; l++) {
                const u64* o = sm + ((size_t)(l * wc + t) * nslots + k) * 2;
                s = gl::e2_add(s, gl::e2_make(o[0], o[1]));
            }
            u64* o = p.partial + (((u64)blockIdx.x * wc + t) * nslots + k) * 2;
            o[0] = s.a;
            o[1] = s.b;
        }
    }
}

// sums[e] = sum over the CTAs of partial[cta][e], e over (column, slot): the host then sees W * (npts + 1) extension values
// per matrix instead of one set per CTA (at 2^16 rows the host-side sum over 592 CTAs cost more than the kernels).
// One warp per element: the lanes stride over the CTAs and combine with shuffles (a single thread walking ~900 partials is a
// 900-deep chain of dependent loads: 0.30 ms per proof at 2^20 rows).
__global__ void __launch_bounds__(128) k_bary_sum(const u64* partial, u32 ctas, u32 n, u64* sums) {
    const u32 e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (e >= n) return;
    gl::e2 s = gl::e2_make(0, 0);
    for (u32 b = lane; b < ctas; b += 32) {
        const u64* o = partial + ((size_t)b * n + e) * 2;
        s = gl::e2_add(s, gl::e2_make(o[0], o[1]));
    }
    for (int d = 16; d >= 1; d >>= 1) {
        u64 oa = __shfl_xor_sync(0xffffffffu, s.a, d), ob = __shfl_xor_sync(0xffffffffu, s.b, d);
        s = gl::e2_add(s, gl::e2_make(oa, ob));
    }
    if (lane == 0) {
        sums[2 * (size_t)e] = s.a;
        sums[2 * (size_t)e + 1] = s.b;
    }
}

// ro[i] += sum_p aoff_p * (yred_p - Mred_i) * invden_p[i],  Mred_i = sum_c alpha^c M[i][c]
struct ReduceParams {
    const u64* M;
    const u64* apow;  // w x 2
    const u64* invden[kMaxPts];
    u64* ro;
    u64 H;        // local rows of M
    u64 ro_off;   // ro index of local row 0 (the FRI owner of a sharded opening keeps the full-length vector)
    u64 aoff[kMaxPts][2], yred[kMaxPts][2];
    u32 w, npts, tile_rows;
};
constexpr int kRedThreads = 128;
constexpr size_t kRedMaxSmem = 200 * 1024;
// rows per tile: the largest power of two <= 128 whose tile fits 64 KB; at least 4 so that the lanes sharing a row
// (128 / tile_rows <= 32) sit in one warp
static u32 reduce_tile_rows(u64 w) {
    u32 tr = 128;
    while (tr > 4 && (size_t)tr * (w | 1) * 8 > 64 * 1024) tr >>= 1;
    return tr;
}
// the tile plus the w alpha powers; within kRedMaxSmem up to 4266 columns (4 * 4267 + 2 * 4266 = 25,600 u64)
static size_t reduce_smem(u64 w) { return ((size_t)reduce_tile_rows(w) * (w | 1) + 2 * w) * 8; }
// A tile of tile_rows rows (power of two <= 128) is staged in shared memory; 128 / tile_rows lanes share a row, each
// accumulating the columns c = lane (mod lanes) lazily; the lanes' partial dot products are combined with shuffles.
__global__ void __launch_bounds__(kRedThreads) k_reduce_openings(ReduceParams p) {
    extern __shared__ u64 sm_r[];
    const u32 TR = p.tile_rows, tpr = kRedThreads / TR;
    const u32 pitch = p.w | 1;
    u64* tile = sm_r;                     // [TR][pitch]
    u64* ap = sm_r + (size_t)TR * pitch;  // [w][2]
    const u64 row0 = (u64)blockIdx.x * TR;
    const u32 nrows = (u32)min((u64)TR, p.H - row0);
    for (u32 e = threadIdx.x; e < 2 * p.w; e += blockDim.x) ap[e] = p.apow[e];
    const u64* src = p.M + row0 * p.w;
    if (p.w == pitch) {
        for (u32 e = threadIdx.x; e < nrows * p.w; e += blockDim.x) tile[e] = src[e];
    } else {
        // (row, column) of element e is advanced without a division per element
        u32 rr = threadIdx.x / p.w, cc = threadIdx.x % p.w;
        const u32 dr = kRedThreads / p.w, dc = kRedThreads % p.w;
        for (u32 e = threadIdx.x; e < nrows * p.w; e += kRedThreads) {
            tile[rr * pitch + cc] = src[e];
            rr += dr;
            cc += dc;
            if (cc >= p.w) { cc -= p.w; rr++; }
        }
    }
    __syncthreads();
    const u32 r = threadIdx.x / tpr, lane = threadIdx.x % tpr;  // tpr divides 32: a row's lanes sit in one warp
    const bool live = r < nrows;
    gl::Acc160 a0 = gl::acc_zero(), a1 = gl::acc_zero();
    if (live) {
        const u64* row = tile + (size_t)r * pitch;
        for (u32 c = lane; c < p.w; c += tpr) {
            u64 v = row[c];
            gl::acc_mac(a0, v, ap[2 * c]);
            gl::acc_mac(a1, v, ap[2 * c + 1]);
        }
    }
    u64 m0 = gl::acc_reduce(a0), m1 = gl::acc_reduce(a1);
    for (u32 d = 1; d < tpr; d <<= 1) {  // tpr is a power of two <= 32 (tile_rows >= 4) or the row spans whole warps
        u64 o0 = __shfl_xor_sync(0xffffffffu, m0, d), o1 = __shfl_xor_sync(0xffffffffu, m1, d);
        m0 = gl::add(m0, o0);
        m1 = gl::add(m1, o1);
    }
    if (!live || lane != 0) return;
    const u64 i = row0 + r, io = p.ro_off + i;
    gl::e2 acc = gl::e2_make(p.ro[2 * io], p.ro[2 * io + 1]);
    for (u32 k = 0; k < p.npts; k++) {
        gl::e2 diff = gl::e2_make(gl::sub(p.yred[k][0], m0), gl::sub(p.yred[k][1], m1));
        gl::e2 d = gl::e2_make(p.invden[k][2 * i], p.invden[k][2 * i + 1]);
        gl::e2 t = gl::e2_mul(gl::e2_mul(gl::e2_make(p.aoff[k][0], p.aoff[k][1]), diff), d);
        acc = gl::e2_add(acc, t);
    }
    p.ro[2 * io] = acc.a;
    p.ro[2 * io + 1] = acc.b;
}

// dst[i] += src[i] over n extension elements (shards of reduced openings added into the FRI owner's vector)
__global__ void __launch_bounds__(256) k_ext_add(u64* dst, const u64* src, u64 n) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * n) return;
    dst[i] = gl::add(dst[i], src[i]);
}
// v[i] += c over n extension elements (the running-sum offset of a row block of a stage-2 trace)
__global__ void __launch_bounds__(256) k_ext_add_scalar(u64* v, u64 n, gl::e2 cst) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * n) return;
    v[i] = gl::add(v[i], (i & 1) ? cst.b : cst.a);
}

// ---- the commit phase's transcript on the device ---------------------------------------------------------------------------
// One FRI round of the reference's challenger (`DeterministicPow<SerializingChallenger64<Goldilocks, HashChallenger<u8, Blake3,
// 32>>>`, src/types.rs:28-81) when commit_proof_of_work_bits = 0 (`grind(0)` touches nothing):
//     observe(root): input = input || root, output buffer cleared        sample_algebra_element(): flush = BLAKE3(input),
//     input := digest, output := digest; bytes are popped from the END, 8 per u64 (first popped = least significant),
//     rejection-sampled below p, coordinate 0 first; when the four candidates of a digest run out the next flush hashes the
//     32-byte input again.
// The input buffer is the 32-byte digest of the previous flush (state) in every round but the first, whose buffer (`prefix`, at
// most 960 bytes: one BLAKE3 chunk with the root) the host hands over. The host replays the same steps on its own challenger
// afterwards (host/gpu_backend.hpp) and compares every beta.
struct FriChal {
    gl::e2 half_beta, beta_sq, beta;
};
__device__ __forceinline__ u32 bswap32(u32 x) { return __byte_perm(x, 0, 0x0123); }
__device__ __noinline__ void fri_challenge_step(const uint8_t* prefix, u32 prefix_len, u32* state, const u32* root, FriChal* out,
                                                u32* root_out) {
    const u32 plen = prefix ? prefix_len : 32u, total = plen + 32u;
    const uint8_t* pre = prefix ? prefix : reinterpret_cast<const uint8_t*>(state);
    const uint8_t* rb = reinterpret_cast<const uint8_t*>(root);
    u32 cv[8];
    b3::set_iv(cv);
    const u32 nblocks = (total + 63u) / 64u;
    for (u32 b = 0; b < nblocks; b++) {
        u32 m[16];
#pragma unroll
        for (int i = 0; i < 16; i++) {
            u32 w = 0;
            for (int k = 0; k < 4; k++) {
                const u32 pos = b * 64u + 4u * i + k;
                u32 byte = pos < plen ? pre[pos] : pos < total ? rb[pos - plen] : 0u;
                w |= byte << (8 * k);
            }
            m[i] = w;
        }
        const u32 blen = min(64u, total - b * 64u);
        const u32 flags = (b == 0 ? b3::CHUNK_START : 0u) | (b + 1 == nblocks ? (b3::CHUNK_END | b3::ROOT) : 0u);
        b3::compress<false>(cv, m, 0, 0, blen, flags);
    }
    u64 coord[2];
    int got = 0;
    for (;;) {
        for (int cnd = 0; cnd < 4 && got < 2; cnd++) {
            const u64 v = ((u64)bswap32(cv[6 - 2 * cnd]) << 32) | bswap32(cv[7 - 2 * cnd]);
            if (v < GLD_P) coord[got++] = v;
        }
        if (got == 2) break;
        u32 m[16] = {cv[0], cv[1], cv[2], cv[3], cv[4], cv[5], cv[6], cv[7], 0, 0, 0, 0, 0, 0, 0, 0};
        b3::set_iv(cv);
        b3::compress<false>(cv, m, 0, 0, 32, b3::CHUNK_START | b3::CHUNK_END | b3::ROOT);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) { state[i] = cv[i]; root_out[i] = root[i]; }
    const gl::e2 beta = gl::e2_make(coord[0], coord[1]);
    out->beta = beta;
    out->half_beta = gl::e2_make(gl::halve(beta.a), gl::halve(beta.b));
    out->beta_sq = gl::e2_mul(beta, beta);
}
__global__ void k_fri_challenge(const uint8_t* prefix, u32 prefix_len, u32* state, const u32* root, FriChal* out, u32* root_out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) fri_challenge_step(prefix, prefix_len, state, root, out, root_out);
}

// out[i] = (lo + hi)/2 + (beta/2) * g^{-rev(i)} * (lo - hi)  [+ beta^2 * roll[i]],  (lo, hi) = in[2i], in[2i+1]
// `chal` (device) overrides the by-value challenge when the transcript runs on the device.
__global__ void __launch_bounds__(256) k_fri_fold(const u64* in, u64* out, u64 half_len, u32 log_half, gl::e2 half_beta,
                                                  gl::PowTable ginv_tab, const u64* roll, gl::e2 beta_sq, const FriChal* chal) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= half_len) return;
    if (chal) { half_beta = chal->half_beta; beta_sq = chal->beta_sq; }
    gl::e2 lo = gl::e2_make(in[4 * i], in[4 * i + 1]), hi = gl::e2_make(in[4 * i + 2], in[4 * i + 3]);
    gl::e2 s = gl::e2_add(lo, hi), d = gl::e2_sub(lo, hi);
    s = gl::e2_make(gl::halve(s.a), gl::halve(s.b));
    u64 gp = gl::pow_lookup(ginv_tab, gl::rev_bits((u32)i, log_half));
    gl::e2 t = gl::e2_mul_base(gl::e2_mul(half_beta, d), gp);
    gl::e2 r = gl::e2_add(s, t);
    if (roll) r = gl::e2_add(r, gl::e2_mul(beta_sq, gl::e2_make(roll[2 * i], roll[2 * i + 1])));
    out[2 * i] = r.a;
    out[2 * i + 1] = r.b;
}

// Small commit-phase rounds in ONE launch of one CTA: fold the committed vector (as k_fri_fold), hash the rows of the folded
// vector (2 extension elements = 32 bytes = one BLAKE3 block) and build every node layer through shared memory. Replaces
// k_fri_fold + k_hash_rows_staged + k_merkle_subtree of the NEXT round for vectors of at most kFusedFoldMax elements: the
// tail of the commit phase is latency, not work (a dozen rounds of ~8 us kernels each waiting for a root read-back).
constexpr u32 kFusedFoldMax = 4096;  // folded length; rows = 2048 -> 64 KB + 32 KB of shared memory
struct FoldCommitParams {
    const u64* in;
    u64* out;
    const u64* roll;
    uint4* digests;          // all layers back to back
    u64 layer_off[13];
    gl::e2 half_beta, beta_sq;
    gl::PowTable ginv_tab;
    u32 half_len, log_half, n_layers;
    const FriChal* chal;      // device-side transcript: this round's challenge (overrides half_beta / beta_sq), or null
    u32* fs_state;            // device-side transcript: challenger state, advanced with the new root when chal_next != null
    FriChal* chal_next;       // where the NEXT round's challenge goes
    u32* root_out;            // 8 words: copy of the new root for the host
};
__device__ __forceinline__ gl::e2 fold_one(const FoldCommitParams& p, gl::e2 half_beta, gl::e2 beta_sq, u32 i) {
    gl::e2 lo = gl::e2_make(p.in[4 * i], p.in[4 * i + 1]), hi = gl::e2_make(p.in[4 * i + 2], p.in[4 * i + 3]);
    gl::e2 s = gl::e2_add(lo, hi), d = gl::e2_sub(lo, hi);
    s = gl::e2_make(gl::halve(s.a), gl::halve(s.b));
    u64 gp = gl::pow_lookup(p.ginv_tab, gl::rev_bits(i, p.log_half));
    gl::e2 r = gl::e2_add(s, gl::e2_mul_base(gl::e2_mul(half_beta, d), gp));
    if (p.roll) r = gl::e2_add(r, gl::e2_mul(beta_sq, gl::e2_make(p.roll[2 * i], p.roll[2 * i + 1])));
    return r;
}
__global__ void __launch_bounds__(256) k_fri_fold_commit(const __grid_constant__ FoldCommitParams p) {
    extern __shared__ uint4 sm_f[];
    const u32 rows = p.half_len >> 1;
    uint4* bufA = sm_f;             // rows digests
    uint4* bufB = sm_f + 2 * rows;  // rows / 2 digests
    const gl::e2 hb = p.chal ? p.chal->half_beta : p.half_beta, bsq = p.chal ? p.chal->beta_sq : p.beta_sq;
    for (u32 j = threadIdx.x; j < rows; j += blockDim.x) {
        gl::e2 a = fold_one(p, hb, bsq, 2 * j), b = fold_one(p, hb, bsq, 2 * j + 1);
        p.out[4 * j] = a.a; p.out[4 * j + 1] = a.b; p.out[4 * j + 2] = b.a; p.out[4 * j + 3] = b.b;
        u32 m[16] = {(u32)a.a, (u32)(a.a >> 32), (u32)a.b, (u32)(a.b >> 32), (u32)b.a, (u32)(b.a >> 32), (u32)b.b, (u32)(b.b >> 32),
                     0, 0, 0, 0, 0, 0, 0, 0};
        u32 cv[8];
        b3::set_iv(cv);
        b3::compress<false>(cv, m, 0, 0, 32, b3::CHUNK_START | b3::CHUNK_END | b3::ROOT);
        uint4 d0 = make_uint4(cv[0], cv[1], cv[2], cv[3]), d1 = make_uint4(cv[4], cv[5], cv[6], cv[7]);
        bufA[2 * j] = d0; bufA[2 * j + 1] = d1;
        p.digests[2 * (p.layer_off[0] + j)] = d0; p.digests[2 * (p.layer_off[0] + j) + 1] = d1;
    }
    __syncthreads();
    for (u32 l = 1; l < p.n_layers; l++) {
        const u32 nodes = rows >> l;
        const uint4* src = (l & 1) ? bufA : bufB;
        uint4* dst = (l & 1) ? bufB : bufA;
        for (u32 i = threadIdx.x; i < nodes; i += blockDim.x) {
            uint4 a0 = src[4 * i], a1 = src[4 * i + 1], b0 = src[4 * i + 2], b1 = src[4 * i + 3];
            u32 x[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w}, y[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w}, d[8];
            b3::hash_pair(x, y, d);
            uint4 d0 = make_uint4(d[0], d[1], d[2], d[3]), d1 = make_uint4(d[4], d[5], d[6], d[7]);
            dst[2 * i] = d0; dst[2 * i + 1] = d1;
            p.digests[2 * (p.layer_off[l] + i)] = d0; p.digests[2 * (p.layer_off[l] + i) + 1] = d1;
        }
        __syncthreads();
    }
    // device-side transcript: observe the new root, sample the next round's beta (thread 0 wrote the root itself)
    if (p.chal_next && threadIdx.x == 0)
        fri_challenge_step(nullptr, 0, p.fs_state, reinterpret_cast<const u32*>(p.digests + 2 * p.layer_off[p.n_layers - 1]), p.chal_next,
                           p.root_out);
}

}  // namespace msg

struct msgpu_open {
    struct Mat {
        const u64* ptr;
        u64 height, width;   // GLOBAL LDE height
        u32 log_h;
        std::vector<msh::Fp2> points;
        std::vector<std::vector<msh::Fp2>> values;  // [point][column]
        // row shards (msgpu_open_begin_shard): this rank holds stored rows [row0, row0 + rows) of the matrix at `ptr`;
        // rows = 0: the matrix lives elsewhere (shapes only). Unsharded: row0 = 0, rows = height.
        u64 row0 = 0, rows = 0;
    };
    msg::Ctx* ctx = nullptr;
    u32 log_blowup = 0;
    bool sharded = false, fri_owner = true;
    std::vector<std::vector<Mat>> rounds;
    struct InvDen {
        msh::Fp2 z;
        u32 log_h;
        msg::DevBuf buf;
        u64 row0 = 0, len = 0;
    };
    // sharded evaluation: the barycentric sums of the local rows, to be summed over the ranks before the values exist
    struct PendingSum {
        size_t round, mat, sums_off;
        u32 npts, c0, wc;
        size_t p0;
    };
    std::vector<PendingSum> pending_sums;
    std::vector<u64> raw_sums;
    std::vector<InvDen> invdens;
    u64 n_values = 0;
    // FRI
    struct Input {
        u64* ptr;
        u64 len;
        msg::DevBuf own;  // empty once the commit phase has taken the input over (input 0: `cur_own`) or rolled it in
    };
    std::vector<Input> inputs;  // tallest first
    size_t next_input = 0;
    u64* cur = nullptr;
    u64 cur_len = 0;
    msg::DevBuf cur_own;         // holds `cur` until it is committed (then its layer holds it) or built ahead into `pending`
    bool cur_committed = false;  // the protocol: a vector is committed before it is folded, and folded before the next commit
    std::vector<std::unique_ptr<msgpu_pdata>> layers;
    std::unique_ptr<msgpu_pdata> pending;  // layer over `cur` built ahead by the fused fold; adopted by the next commit_round
    bool pending_has_chal = false;         // the fused fold that built `pending` also ran the transcript step for its root
};

namespace msg {

static gl::PowTable lde_x_table(Ctx& c, u32 log_h) {
    return c.pow_table(msh::two_adic_generator(log_h).v, msh::GL_GENERATOR, log_h).view();
}

// Unsharded: one array per point at the largest height opened there serves every shorter matrix (its first rows are the
// shorter domain). Sharded: one array per (point, height, row range), since a shard of a shorter matrix is not a prefix.
static u64* find_invden(msgpu_open* op, const msh::Fp2& z, const msgpu_open::Mat& m) {
    for (auto& d : op->invdens) {
        if (!(d.z == z)) continue;
        if (!op->sharded && d.log_h >= m.log_h) return d.buf.u();
        if (op->sharded && d.log_h == m.log_h && d.row0 == m.row0 && d.len == m.rows) return d.buf.u();
    }
    throw Error(-3, "open: missing inverse denominators");
}

// The tallest input is the first vector of the commit phase; the shorter ones are rolled into the folds of their height.
static void start_commit_phase(msgpu_open* op) {
    std::sort(op->inputs.begin(), op->inputs.end(), [](const msgpu_open::Input& a, const msgpu_open::Input& b) { return a.len > b.len; });
    op->cur = op->inputs[0].ptr;
    op->cur_len = op->inputs[0].len;
    op->cur_own = std::move(op->inputs[0].own);
    op->next_input = 1;
    op->cur_committed = false;
}

// values from the barycentric sums (S1, S2 per column and point): y = (z * S2 - S1) * (z^h - g^h) / (h * g^h), g = GENERATOR
static void finish_values(msgpu_open* op, const u64* sums) {
    for (auto& ps : op->pending_sums) {
        auto& m = op->rounds[ps.round][ps.mat];
        u32 log_h = m.log_h - op->log_blowup;
        msh::Fp shift_pow = msh::Fp(msh::GL_GENERATOR).exp_power_of_2(log_h);
        msh::Fp denom_inv = (shift_pow * msh::Fp((msh::u64)1 << log_h)).inverse();
        const u32 nslots = ps.npts + 1;
        msh::Fp2 scale[kMaxPts];
        for (u32 k = 0; k < ps.npts; k++) scale[k] = (m.points[ps.p0 + k].exp_power_of_2(log_h) - shift_pow) * denom_inv;
        const u64* hs = sums + ps.sums_off;
        for (u32 cc = 0; cc < ps.wc; cc++) {
            msh::Fp s1 = msh::Fp(hs[((size_t)cc * nslots) * 2]);
            for (u32 k = 0; k < ps.npts; k++) {
                size_t o = ((size_t)cc * nslots + k + 1) * 2;
                msh::Fp2 s2 = msh::Fp2(msh::Fp((msh::u64)hs[o]), msh::Fp((msh::u64)hs[o + 1]));
                m.values[ps.p0 + k][ps.c0 + cc] = (m.points[ps.p0 + k] * s2 - s1) * scale[k];
            }
        }
    }
    op->pending_sums.clear();
}

static void evaluate_all(Ctx& c, msgpu_open* op) {
    StageScope ss(c, "open");
    // 1. inverse denominators per distinct point: unsharded at the largest LDE height opened there; sharded per
    //    (point, height, row range) of the rows this rank holds
    for (auto& round : op->rounds)
        for (auto& m : round) {
            if (m.rows == 0) continue;
            for (auto& z : m.points) {
                bool found = false;
                for (auto& d : op->invdens) {
                    if (!(d.z == z)) continue;
                    if (!op->sharded) { d.log_h = std::max(d.log_h, m.log_h); d.len = 1ull << d.log_h; found = true; }
                    else if (d.log_h == m.log_h && d.row0 == m.row0 && d.len == m.rows) found = true;
                }
                if (!found) op->invdens.push_back(msgpu_open::InvDen{z, m.log_h, DevBuf(), m.row0, m.rows});
            }
        }
    for (auto& d : op->invdens) {
        d.buf = DevBuf(c, d.len * 16);
        u64 threads = (d.len + kInvPerThread - 1) / kInvPerThread;
        launch(c, "k_inv_denoms", k_inv_denoms, (unsigned)((threads + 255) / 256), 256, 0, d.buf.u(), d.log_h, gl::e2{d.z.c[0].v, d.z.c[1].v},
               lde_x_table(c, d.log_h), d.row0, d.len);
    }
    // 2. barycentric sums per matrix (all of its points in one pass over the low coset = the first height >> log_blowup stored
    //    rows; a shard contributes the part of them it holds)
    std::vector<DevBuf> partials;
    size_t sums_total = 0;
    for (auto& round : op->rounds)
        for (auto& m : round)
            for (size_t p0 = 0; p0 < m.points.size(); p0 += kMaxPts)
                sums_total += m.width * (std::min<size_t>(kMaxPts, m.points.size() - p0) + 1) * 2;
    DevBuf d_sums(c, std::max<size_t>(sums_total, 1) * 8);
    MSG_CUDA(cudaMemsetAsync(d_sums.p, 0, std::max<size_t>(sums_total, 1) * 8, c.stream));
    size_t sums_off = 0;
    op->pending_sums.clear();
    for (size_t ri = 0; ri < op->rounds.size(); ri++)
        for (size_t mi = 0; mi < op->rounds[ri].size(); mi++) {
            auto& m = op->rounds[ri][mi];
            m.values.assign(m.points.size(), std::vector<msh::Fp2>(m.width));
            if (m.width == 0) continue;
            const u64 h_all = m.height >> op->log_blowup;
            const u64 h = m.row0 >= h_all ? 0 : std::min<u64>(m.rows, h_all - m.row0);  // local rows inside the low coset
            for (size_t p0 = 0; p0 < m.points.size(); p0 += kMaxPts) {
                u32 npts = (u32)std::min<size_t>(kMaxPts, m.points.size() - p0);
                for (u32 c0 = 0; c0 < m.width; c0 += 256) {
                    BaryParams bp{};
                    bp.M = m.ptr;
                    bp.h = h;
                    bp.w = (u32)m.width;
                    bp.c0 = c0;
                    bp.wc = (u32)std::min<u64>(256, m.width - c0);
                    bp.rows_per_step = 256 / bp.wc;
                    op->pending_sums.push_back(msgpu_open::PendingSum{ri, mi, sums_off, npts, c0, bp.wc, p0});
                    const size_t my_off = sums_off;
                    sums_off += (size_t)bp.wc * (npts + 1) * 2;
                    if (h == 0) continue;  // nothing of the low coset here: the sums stay zero
                    for (u32 k = 0; k < npts; k++) bp.invden[k] = find_invden(op, m.points[p0 + k], m);
                    bp.tile_rows = (u32)std::min<u64>(256, std::max<u64>(8, 4096 / bp.wc));
                    u64 want = (h + bp.tile_rows - 1) / bp.tile_rows;
                    u32 ctas = (u32)std::min<u64>(want, (u64)c.sm_count * 6);
                    partials.emplace_back(c, (size_t)ctas * bp.wc * (npts + 1) * 16);
                    bp.partial = partials.back().u();
                    // at most 46,448 bytes when the dd tile is padded (wc = 19, tile_rows = 215, 4 points) and 49,152 without
                    // (wc = 16, tile_rows = 256, 4 points): both within the default dynamic shared memory limit
                    size_t smem = std::max((size_t)bp.rows_per_step * bp.wc * (npts + 1) * 16,
                                           (bary_dd_offset(bp.tile_rows, bp.wc) + (size_t)bp.tile_rows * npts * 2) * 8);
                    switch (npts) {
                        case 1: launch(c, "k_bary_partial", k_bary_partial<1>, ctas, 256, smem, bp); break;
                        case 2: launch(c, "k_bary_partial", k_bary_partial<2>, ctas, 256, smem, bp); break;
                        case 3: launch(c, "k_bary_partial", k_bary_partial<3>, ctas, 256, smem, bp); break;
                        default: launch(c, "k_bary_partial", k_bary_partial<4>, ctas, 256, smem, bp); break;
                    }
                    const u32 n = bp.wc * (npts + 1);
                    launch(c, "k_bary_sum", k_bary_sum, (n * 32 + 127) / 128, 128, 0, bp.partial, ctas, n, d_sums.u() + my_off);
                }
            }
        }
    op->raw_sums.assign(std::max<size_t>(sums_total, 1), 0);
    if (sums_total) MSG_CUDA(cudaMemcpyAsync(op->raw_sums.data(), d_sums.p, sums_total * 8, cudaMemcpyDeviceToHost, c.stream));  // ONE read-back
    c.sync();
    op->raw_sums.resize(sums_total);
    // sharded: the sums of all ranks are added first (msgpu_open_sums / msgpu_open_finish_values)
    if (!op->sharded) finish_values(op, op->raw_sums.data());
}

static void reduce_all(Ctx& c, msgpu_open* op, msh::Fp2 alpha) {
    StageScope ss(c, "open");
    // checked before anything is allocated or copied, so that a refused opening leaves nothing behind
    for (auto& round : op->rounds)
        for (auto& m : round)
            MSG_REQUIRE(m.points.empty() || m.rows == 0 || reduce_smem(m.width) <= kRedMaxSmem,
                        "open: matrix too wide for the reduced-openings kernel (more than 4266 columns)");
    size_t max_w = 1;
    for (auto& round : op->rounds)
        for (auto& m : round) max_w = std::max<size_t>(max_w, m.width);
    std::vector<msh::Fp2> apow(max_w);
    msh::Fp2 acc = msh::Fp2::one();
    for (size_t i = 0; i < max_w; i++) { apow[i] = acc; acc *= alpha; }
    std::vector<u64> apow_flat(2 * max_w);
    for (size_t i = 0; i < max_w; i++) { apow_flat[2 * i] = apow[i].c[0].v; apow_flat[2 * i + 1] = apow[i].c[1].v; }
    DevBuf d_apow(c, apow_flat.size() * 8);
    MSG_CUDA(cudaMemcpyAsync(d_apow.p, apow_flat.data(), apow_flat.size() * 8, cudaMemcpyHostToDevice, c.stream));
    DevBuf ro[33];
    u64 ro_len[33] = {0};
    u64 num_reduced[33] = {0};
    ensure_max_smem(k_reduce_openings, (int)kRedMaxSmem);
    for (auto& round : op->rounds)
        for (auto& m : round) {
            u32 lh = m.log_h;
            // the FRI owner keeps full-length vectors (the other ranks' shards are added into them); another rank only the
            // rows it holds, and nothing for heights it has no rows of
            const bool full = !op->sharded || op->fri_owner;
            if (!ro[lh] && (full || m.rows)) {  // p3 creates the height's vector for every matrix of every round, opened or not
                ro_len[lh] = full ? m.height : m.rows;
                ro[lh] = DevBuf(c, ro_len[lh] * 16);
                MSG_CUDA(cudaMemsetAsync(ro[lh].p, 0, ro_len[lh] * 16, c.stream));
            }
            if (m.points.empty()) continue;
            if (m.rows == 0) {  // lives elsewhere: only the alpha-power counter of its height advances
                num_reduced[lh] += m.width * m.points.size();
                continue;
            }
            MSG_REQUIRE(full || ro_len[lh] == m.rows, "open_reduce: shards of one height must cover the same rows");
            for (size_t p0 = 0; p0 < m.points.size(); p0 += kMaxPts) {
                u32 npts = (u32)std::min<size_t>(kMaxPts, m.points.size() - p0);
                ReduceParams rp{};
                rp.M = m.ptr;
                rp.apow = d_apow.u();
                rp.ro = ro[lh].u();
                rp.H = m.rows;
                rp.ro_off = full ? m.row0 : 0;
                rp.w = (u32)m.width;
                rp.npts = npts;
                for (u32 k = 0; k < npts; k++) {
                    rp.invden[k] = find_invden(op, m.points[p0 + k], m);
                    msh::Fp2 aoff = alpha.pow(num_reduced[lh]);
                    msh::Fp2 yred;
                    for (size_t cc = 0; cc < m.width; cc++) yred += apow[cc] * m.values[p0 + k][cc];
                    rp.aoff[k][0] = aoff.c[0].v; rp.aoff[k][1] = aoff.c[1].v;
                    rp.yred[k][0] = yred.c[0].v; rp.yred[k][1] = yred.c[1].v;
                    num_reduced[lh] += m.width;
                }
                const u32 tr = reduce_tile_rows(m.width);
                rp.tile_rows = tr;
                launch(c, "k_reduce_openings", k_reduce_openings, (unsigned)((m.rows + tr - 1) / tr), kRedThreads, reduce_smem(m.width), rp);
            }
        }
    for (int lh = 32; lh >= 0; lh--)
        if (ro[lh]) op->inputs.push_back(msgpu_open::Input{ro[lh].u(), ro_len[lh], std::move(ro[lh])});
    c.sync();  // apow_flat (pageable) must outlive its copy
    MSG_REQUIRE(!op->inputs.empty(), "open: nothing to open");
    start_commit_phase(op);
}


// One fold of the committed vector. The challenge comes from the host (`beta`) or from device memory (`chal`). With
// fuse_commit and a folded length in [2, kFusedFoldMax] the folded vector is committed by the same launch (op->pending) and,
// when next_state / next_chal are given, the transcript step for that commitment runs in it too.
static void fri_fold_impl(msgpu_open* op, const msh::Fp2* beta, const FriChal* chal, bool fuse_commit, u32* next_state,
                          FriChal* next_chal, u32* next_root_out) {
    Ctx& c = *op->ctx;
    StageScope ss(c, "fri");
    u64 half = op->cur_len / 2;
    u32 log_half = ilog2(half);
    msh::Fp2 hb, bsq;
    if (beta) { hb = beta->halve(); bsq = beta->square(); }
    const u64* roll = nullptr;
    if (op->next_input < op->inputs.size() && op->inputs[op->next_input].len == half) roll = op->inputs[op->next_input].ptr;
    DevBuf out_buf(c, half * 16);
    u64* out = out_buf.u();
    gl::PowTable tab = c.pow_table(msh::two_adic_generator(log_half + 1).inverse().v, 1, log_half + 1).view();
    if (fuse_commit && half >= 2 && half <= kFusedFoldMax) {
        // fold + Merkle commitment of the folded vector (rows of 2 extension elements) in one launch
        auto pd = std::make_unique<msgpu_pdata>();
        const u64 rows = half / 2;
        mmcs_layout_layers(c, pd.get(), rows);
        pd->mats.push_back(msgpu_pdata::Mat{out, rows, 4, std::move(out_buf)});
        pd->total_width = 4;
        FoldCommitParams fp{};
        fp.in = op->cur;
        fp.out = out;
        fp.roll = roll;
        fp.digests = (uint4*)pd->digests.p;
        fp.n_layers = (u32)pd->layer_off.size();
        for (size_t l = 0; l < pd->layer_off.size(); l++) fp.layer_off[l] = pd->layer_off[l];
        fp.half_beta = gl::e2{hb.c[0].v, hb.c[1].v};
        fp.beta_sq = gl::e2{bsq.c[0].v, bsq.c[1].v};
        fp.ginv_tab = tab;
        fp.half_len = (u32)half;
        fp.log_half = log_half;
        fp.chal = chal;
        fp.fs_state = next_state;
        fp.chal_next = next_chal;
        fp.root_out = next_root_out;
        ensure_max_smem(k_fri_fold_commit, (int)(kFusedFoldMax / 2 * 48));
        launch(c, "k_fri_fold_commit", k_fri_fold_commit, 1, 256, (size_t)rows * 48, fp);
        if (!chal) MSG_CUDA(cudaMemcpyAsync(pd->root, pd->digests.bytes() + pd->layer_off.back() * 32, 32, cudaMemcpyDeviceToHost, c.stream));
        op->pending = std::move(pd);
        op->pending_has_chal = next_chal != nullptr;
    } else {
        launch(c, "k_fri_fold", k_fri_fold, (unsigned)((half + 255) / 256), 256, 0, op->cur, out, half, log_half,
               gl::e2{hb.c[0].v, hb.c[1].v}, tab, roll, gl::e2{bsq.c[0].v, bsq.c[1].v}, chal);
        op->cur_own = std::move(out_buf);
    }
    if (roll) {
        op->inputs[op->next_input].own.reset();
        op->next_input++;
    }
    op->cur = out;
    op->cur_len = half;
    op->cur_committed = false;
}

// shared by msgpu_open_begin / msgpu_open_begin_shard. modes[r] (sharded only): 0 = the round's matrices are here in full
// (e.g. the quotient commitment on the rank that built it), 1 = this rank holds row shard `shard` of `n_shards` of every matrix
// (the prover data holds the SHARDS: heights are 1 / n_shards of the matrices'), 2 = the round lives elsewhere (a placeholder
// prover data carries the shapes).
static void open_begin_impl(msgpu_ctx* h, uint64_t n_rounds, const msgpu_pdata* const* pds, const uint32_t* modes, uint32_t shard,
                            uint32_t n_shards, int fri_owner, const uint64_t* n_points, const uint64_t* points, uint32_t log_blowup,
                            msgpu_open** out, uint64_t* n_values) {
    Ctx& c = h->c;
    MSG_REQUIRE(pds && out && n_values, "open_begin: null argument");
    auto op = std::make_unique<msgpu_open>();
    op->ctx = &c;
    op->log_blowup = log_blowup;
    op->sharded = modes != nullptr;
    op->fri_owner = fri_owner != 0;
    size_t mi = 0, pi = 0;
    u64 total = 0;
    const msh::Fp gen_inv = msh::Fp(msh::GL_GENERATOR).inverse();
    for (u64 r = 0; r < n_rounds; r++) {
        MSG_REQUIRE(pds[r], "open_begin: null prover data");
        const u32 mode = modes ? modes[r] : 0;
        MSG_REQUIRE(mode <= 2, "open_begin: bad round mode");
        std::vector<msgpu_open::Mat> round;
        for (auto& pm : pds[r]->mats) {
            const u64 gh = mode == 1 ? pm.height * n_shards : pm.height;
            msgpu_open::Mat m{pm.ptr, gh, pm.width, ilog2(gh), {}, {}};
            m.rows = mode == 2 ? 0 : pm.height;
            m.row0 = mode == 1 ? (u64)shard * pm.height : 0;
            MSG_REQUIRE(mode == 2 || pm.ptr || pm.width == 0, "open_begin: prover data without matrices (a placeholder needs mode 2)");
            MSG_REQUIRE(m.log_h >= log_blowup, "open_begin: committed matrix shorter than the blowup");
            u64 np = n_points[mi++];
            for (u64 k = 0; k < np; k++, pi++) {
                MSG_REQUIRE(points[2 * pi] < GLD_P && points[2 * pi + 1] < GLD_P, "open_begin: point is not canonical");
                // 1 / (z - x) has no value at a point x of the LDE coset GENERATOR * H; k_inv_denoms inverts in batches, so
                // such a z would silently zero every inverse of its batch. Only a base-field z can lie on the coset.
                MSG_REQUIRE(points[2 * pi + 1] != 0 || (msh::Fp(points[2 * pi]) * gen_inv).exp_power_of_2(m.log_h) != msh::Fp::one(),
                            "open_begin: point lies on the committed LDE coset");
                m.points.push_back(msh::Fp2(msh::Fp(points[2 * pi]), msh::Fp(points[2 * pi + 1])));
            }
            total += np * pm.width;
            round.push_back(std::move(m));
        }
        op->rounds.push_back(std::move(round));
    }
    op->n_values = total;
    evaluate_all(c, op.get());
    *n_values = total;
    *out = op.release();
}

}  // namespace msg

using namespace msg;

extern "C" {

int msgpu_open_begin(msgpu_ctx* h, uint64_t n_rounds, const msgpu_pdata* const* pds, const uint64_t* n_points,
                     const uint64_t* points, uint32_t log_blowup, msgpu_open** out, uint64_t* n_values) {
    return guard([&] { open_begin_impl(h, n_rounds, pds, nullptr, 0, 1, 1, n_points, points, log_blowup, out, n_values); });
}

// ---- Pcs::open over ROW SHARDS (one proof over several GPUs) -----------------------------------------------------------------
int msgpu_open_begin_shard(msgpu_ctx* h, uint64_t n_rounds, const msgpu_pdata* const* pds, const uint32_t* modes, uint32_t shard,
                           uint32_t n_shards, int fri_owner, const uint64_t* n_points, const uint64_t* points, uint32_t log_blowup,
                           msgpu_open** out, uint64_t* n_values, uint64_t* n_sums) {
    return guard([&] {
        MSG_REQUIRE(modes && n_sums && n_shards >= 1 && shard < n_shards && is_pow2(n_shards), "open_begin_shard: bad argument");
        open_begin_impl(h, n_rounds, pds, modes, shard, n_shards, fri_owner, n_points, points, log_blowup, out, n_values);
        *n_sums = (*out)->raw_sums.size();
    });
}
int msgpu_open_sums(msgpu_open* op, uint64_t* out) {
    return guard([&] {
        MSG_REQUIRE(op && op->sharded && (out || op->raw_sums.empty()), "open_sums: not a sharded opening");
        if (!op->raw_sums.empty()) memcpy(out, op->raw_sums.data(), op->raw_sums.size() * 8);
    });
}
int msgpu_open_finish_values(msgpu_open* op, const uint64_t* total_sums) {
    return guard([&] {
        MSG_REQUIRE(op && op->sharded && !op->pending_sums.empty() && (total_sums || op->raw_sums.empty()), "open_finish_values: nothing pending");
        for (size_t i = 0; i < op->raw_sums.size(); i++) MSG_REQUIRE(total_sums[i] < GLD_P, "open_finish_values: sum is not canonical");
        finish_values(op, (const u64*)total_sums);
    });
}
// prover data that carries shapes only (a round whose matrices live on other ranks)
int msgpu_pdata_placeholder(msgpu_ctx* h, uint64_t n_mats, const uint64_t* heights, const uint64_t* widths, msgpu_pdata** out) {
    return guard([&] {
        MSG_REQUIRE(out && n_mats > 0 && heights && widths, "pdata_placeholder: bad argument");
        auto pd = std::make_unique<msgpu_pdata>();
        for (u64 i = 0; i < n_mats; i++) {
            MSG_REQUIRE(is_pow2(heights[i]), "pdata_placeholder: heights must be powers of two");
            pd->mats.push_back(msgpu_pdata::Mat{nullptr, heights[i], widths[i]});
            pd->total_width += widths[i];
            pd->max_height = std::max<u64>(pd->max_height, heights[i]);
        }
        memset(pd->root, 0, 32);
        *out = pd.release();
    });
}
// dst[i] += src[i] / v[i] += c over n extension elements (device pointers)
int msgpu_ext_add_dev(msgpu_ctx* h, uint64_t* dst, const uint64_t* src, uint64_t n) {
    return guard([&] {
        Ctx& c = h->c;
        if (n == 0) return;
        launch(c, "k_ext_add", k_ext_add, (unsigned)((2 * n + 255) / 256), 256, 0, (u64*)dst, (const u64*)src, n);
    });
}
int msgpu_ext_add_scalar_dev(msgpu_ctx* h, uint64_t* v, uint64_t n, const uint64_t* c2) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(c2 && c2[0] < GLD_P && c2[1] < GLD_P, "ext_add_scalar: constant is not canonical");
        if (n == 0) return;
        launch(c, "k_ext_add_scalar", k_ext_add_scalar, (unsigned)((2 * n + 255) / 256), 256, 0, (u64*)v, n, gl::e2{c2[0], c2[1]});
    });
}

int msgpu_open_values(msgpu_open* op, uint64_t* out) {
    return guard([&] {
        size_t o = 0;
        for (auto& round : op->rounds)
            for (auto& m : round)
                for (auto& pv : m.values)
                    for (auto& v : pv) { out[o++] = v.c[0].v; out[o++] = v.c[1].v; }
    });
}

int msgpu_open_reduce(msgpu_open* op, const uint64_t* alpha2, uint64_t* n_inputs, uint32_t* log_max_height) {
    return guard([&] {
        MSG_REQUIRE(op->inputs.empty(), "open_reduce: already reduced");
        reduce_all(*op->ctx, op, msh::Fp2(msh::Fp(alpha2[0]), msh::Fp(alpha2[1])));
        if (n_inputs) *n_inputs = op->inputs.size();
        if (log_max_height) *log_max_height = ilog2(op->inputs[0].len);
    });
}

int msgpu_open_read_input(msgpu_open* op, uint64_t k, uint64_t* out, uint64_t* len_out) {
    return guard([&] {
        MSG_REQUIRE(k < op->inputs.size() && (k == 0 || k >= op->next_input), "open_read_input: input already consumed");
        Ctx& c = *op->ctx;
        if (len_out) *len_out = op->inputs[k].len;
        if (out) {
            MSG_CUDA(cudaMemcpyAsync(out, op->inputs[k].ptr, op->inputs[k].len * 16, cudaMemcpyDeviceToHost, c.stream));
            c.sync();
        }
    });
}

int msgpu_open_input_dev(msgpu_open* op, uint64_t k, uint64_t** dev_ptr, uint64_t* len_out) {
    return guard([&] {
        MSG_REQUIRE(k < op->inputs.size() && (k == 0 || k >= op->next_input), "open_input_dev: input already consumed");
        if (dev_ptr) *dev_ptr = (uint64_t*)op->inputs[k].ptr;
        if (len_out) *len_out = op->inputs[k].len;
    });
}

int msgpu_open_add_input(msgpu_open* op, uint64_t len, uint64_t** dev_ptr) {
    return guard([&] {
        Ctx& c = *op->ctx;
        MSG_REQUIRE(dev_ptr && is_pow2(len), "open_add_input: bad argument");
        MSG_REQUIRE(op->layers.empty() && !op->cur_committed && op->next_input <= 1, "open_add_input: the commit phase has started");
        for (auto& in : op->inputs) MSG_REQUIRE(in.len != len, "open_add_input: this height already has an input (one height class per rank)");
        DevBuf buf(c, len * 16);
        *dev_ptr = (uint64_t*)buf.p;
        if (op->cur_own) op->inputs[0].own = std::move(op->cur_own);  // the commit phase starts over with the tallest input
        op->inputs.push_back(msgpu_open::Input{buf.u(), len, std::move(buf)});
        start_commit_phase(op);
    });
}

int msgpu_fri_current_len(msgpu_open* op, uint64_t* len) {
    return guard([&] {
        MSG_REQUIRE(op->cur, "fri: open_reduce has not run");
        *len = op->cur_len;
    });
}

int msgpu_fri_commit_round(msgpu_open* op, uint8_t* root32) {
    return guard([&] {
        Ctx& c = *op->ctx;
        StageScope ss(c, "fri");
        MSG_REQUIRE(op->cur && !op->cur_committed, "fri_commit_round: nothing to commit");
        MSG_REQUIRE(op->cur_len >= 2, "fri_commit_round: vector too short to fold");
        op->cur_committed = true;
        if (op->pending) {  // the fused fold has already hashed this vector: wait for its root
            op->layers.push_back(std::move(op->pending));
            c.sync();
            memcpy(root32, op->layers.back()->root, 32);
            return;
        }
        auto pd = std::make_unique<msgpu_pdata>();
        // rows of 2 extension elements = 4 base columns (ExtensionMmcs flattening)
        pd->mats.push_back(msgpu_pdata::Mat{op->cur, op->cur_len / 2, 4, std::move(op->cur_own)});
        op->layers.push_back(std::move(pd));
        mmcs_build(c, op->layers.back().get());
        memcpy(root32, op->layers.back()->root, 32);
    });
}

int msgpu_fri_fold(msgpu_open* op, const uint64_t* beta2) {
    return guard([&] {
        MSG_REQUIRE(op->cur && op->cur_committed, "fri_fold: commit the current vector first");
        msh::Fp2 beta{msh::Fp(beta2[0]), msh::Fp(beta2[1])};
        fri_fold_impl(op, &beta, nullptr, true, nullptr, nullptr, nullptr);
    });
}

// The whole commit phase without a host round trip (commit_proof_of_work_bits = 0): per round commit the vector (the root
// stays on the device), k_fri_challenge derives beta from (challenger state, root), the fold reads it from device memory.
// Rounds of at most kFusedFoldMax elements are ONE launch each (fold + leaf hash + node layers + the next transcript step).
// One synchronisation at the end brings back every root and beta.
int msgpu_fri_commit_phase(msgpu_open* op, const uint8_t* input_buffer, uint64_t input_len, uint64_t stop_len, uint64_t max_rounds,
                           uint8_t* roots_out, uint64_t* betas_out, uint64_t* n_rounds) {
    return guard([&] {
        Ctx& c = *op->ctx;
        StageScope ss(c, "fri");
        MSG_REQUIRE(op->cur && !op->cur_committed && !op->pending, "fri_commit_phase: nothing to commit");
        MSG_REQUIRE(input_buffer && input_len >= 1 && input_len <= 960, "fri_commit_phase: the challenger's input buffer must be 1..960 bytes");
        MSG_REQUIRE(is_pow2(stop_len) && stop_len >= 1 && roots_out && betas_out && n_rounds, "fri_commit_phase: bad argument");
        u64 rounds = 0;
        for (u64 l = op->cur_len; l > stop_len; l >>= 1) rounds++;
        MSG_REQUIRE(rounds <= max_rounds, "fri_commit_phase: output buffers too small");
        *n_rounds = rounds;
        if (rounds == 0) return;
        // device transcript state: [state 32 B][roots 32 B x rounds][FriChal x rounds][prefix]
        const size_t off_roots = 32, off_chal = off_roots + 32 * rounds, off_prefix = off_chal + sizeof(FriChal) * rounds;
        DevBuf fs(c, off_prefix + ((input_len + 15) & ~(size_t)15));
        uint8_t* base = (uint8_t*)fs.p;
        u32* d_state = (u32*)base;
        u32* d_roots = (u32*)(base + off_roots);
        FriChal* d_chal = (FriChal*)(base + off_chal);
        uint8_t* d_prefix = base + off_prefix;
        MSG_CUDA(cudaMemcpyAsync(d_prefix, input_buffer, input_len, cudaMemcpyHostToDevice, c.stream));
        for (u64 k = 0; k < rounds; k++) {
            // commit the current vector (unless the fused fold of the previous round already did, transcript step included)
            bool have_chal = false;
            if (op->pending) {
                op->layers.push_back(std::move(op->pending));
                have_chal = op->pending_has_chal;
                op->pending_has_chal = false;
            } else {
                op->layers.push_back(std::make_unique<msgpu_pdata>());  // ExtensionMmcs rows of 2 elements
                op->layers.back()->mats.push_back(msgpu_pdata::Mat{op->cur, op->cur_len / 2, 4, std::move(op->cur_own)});
            }
            op->cur_committed = true;
            msgpu_pdata* pd = op->layers.back().get();
            if (!pd->digests) mmcs_build_async(c, pd);
            if (!have_chal)
                launch(c, "k_fri_challenge", k_fri_challenge, 1, 32, 0, k == 0 ? d_prefix : nullptr, (u32)input_len, d_state,
                       (const u32*)(pd->digests.bytes() + pd->layer_off.back() * 32), d_chal + k, d_roots + 8 * k);
            const bool last = k + 1 == rounds;
            fri_fold_impl(op, nullptr, d_chal + k, !last, last ? nullptr : d_state, last ? nullptr : d_chal + k + 1,
                          last ? nullptr : d_roots + 8 * (k + 1));
        }
        std::vector<uint8_t> host(32 * rounds + sizeof(FriChal) * rounds);
        MSG_CUDA(cudaMemcpyAsync(host.data(), d_roots, host.size(), cudaMemcpyDeviceToHost, c.stream));
        c.sync();
        memcpy(roots_out, host.data(), 32 * rounds);
        const FriChal* hc = (const FriChal*)(host.data() + 32 * rounds);
        for (u64 k = 0; k < rounds; k++) {
            betas_out[2 * k] = hc[k].beta.a;
            betas_out[2 * k + 1] = hc[k].beta.b;
            memcpy(op->layers[op->layers.size() - rounds + k]->root, roots_out + 32 * k, 32);
        }
    });
}

int msgpu_fri_read_current(msgpu_open* op, uint64_t* out) {
    return guard([&] {
        Ctx& c = *op->ctx;
        MSG_REQUIRE(op->cur, "fri: open_reduce has not run");
        MSG_CUDA(cudaMemcpyAsync(out, op->cur, op->cur_len * 16, cudaMemcpyDeviceToHost, c.stream));
        c.sync();
    });
}

uint64_t msgpu_fri_num_layers(const msgpu_open* op) { return op->layers.size(); }
const msgpu_pdata* msgpu_fri_layer_pdata(const msgpu_open* op, uint64_t layer) {
    return layer < op->layers.size() ? op->layers[layer].get() : nullptr;
}
void msgpu_open_free(msgpu_open* op) { delete op; }

}  // extern "C"
