// Goldilocks NTT / coset low-degree extension kernels (sm_100a).
//
// Replaces, on the device, what the reference obtains from p3-dft `Radix2DitParallel`
// (src/types.rs:200; call sites src/prover.rs:440,650,716) and the `coset_lde_batch(...)
// .bit_reverse_rows()` inside `TwoAdicFriPcs::commit` (src/prover.rs:350,419; src/system.rs:193).
//
// Data layout: row-major n x w matrices of canonical u64, exactly the reference's RowMajorMatrix.
// A transform of size n = 2^L over the rows is split into passes of at most 10 bits. A pass works on
// tiles of T = 2^tb points x 16 adjacent u64 (128-byte row segments, so every global access is a full
// coalesced line) and runs the tb butterfly stages as radix-16 / radix-16 / radix-4 rounds:
//
//   round = one register-resident size-R DFT per thread whose internal twiddles are all POWERS OF TWO
//           (p3's two_adic_generator(k) is 2^96, 2^48, 2^120, 2^156 for k = 1..4, and 2^96 = -1), i.e.
//           multiplications by compile-time constants with zero limbs and free sign flips, followed by ONE
//           general multiplication per element by w_T^{off * r} (Cooley-Tukey / Gentleman-Sande with the
//           twiddles pulled out of the butterflies): 15 general multiplications per 16 elements instead of 32.
//           The twiddles of the round over bits [2, 6) are 64th roots of unity, powers of two as well (2^39 = w_64), so they
//           are shifts too: a 10-bit tile pays ONE general twiddle multiplication per element, in the round over the top
//           bits. DIT tiles run the DIF rounds in mirror order (radix-4 / 16 / 16 from the low bits up) for the same reason.
//   The first round loads straight from global memory into registers and the last round stores straight
//   from registers to global memory (with the inter-pass twiddle folded in), so a tile touches shared
//   memory only between rounds. Thread -> (column, row group) is fixed for the whole kernel: no integer
//   division in any loop.
//
//  * k_ntt_strided: decimation-in-frequency pass over bits [lo, lo+tb) of the row index, natural
//    order in, bit-reversed order out, in place (the 4-step decomposition with the transpose absorbed
//    into index arithmetic). A chain of these is a DFT whose output is stored bit-reversed, which is
//    the storage the reference gets from `dft_batch(..).bit_reverse_rows()`.
//  * k_ntt_block: first pass of the coset evaluation. It reads the bit-reversed coefficients that the
//    inverse transform left behind (contiguous blocks), multiplies row j by shift_s^j / n, runs a
//    decimation-in-time tile (bit-reversed in, natural out) and scatters whole 128-byte row segments to
//    their bit-reversed block. The zero-padded forward transform of size n*B is never materialised: output
//    block rev(s) of n rows is the size-n coset transform with shift * w_{nB}^s (SURVEY Appendix A.3 item 2),
//    so the LDE reads n rows and writes n*B.
//  Inter-pass twiddles and coset scales come from per-size tables built once per context (n entries each,
//  L2-resident while a pass streams): one load + one multiplication per element.
#include "internal.hpp"

namespace msg {

constexpr int kXt = 4;            // tile columns (64-byte row segments); two 512-thread CTAs per SM overlap their load /
                                  // compute / store phases, which one 1024-thread CTA with 16 columns cannot
constexpr int kLogXt = 2;
// Tile rows are kXt u64 (8 words) wide with NO padding; the row index is XOR-swizzled so that the four tile rows a
// half-warp touches in one 64-bit access (4 thread rows x kXt columns) always land in four different 8-word bank groups,
// whichever round is running: rounds address rows that differ in one PAIR of index bits (0-1 for consecutive rows, 2-3 for
// the stride-4 radix-4 round, 4-5 for the stride-16 radix-16 round, ...), and the swizzle folds every pair onto bits 0-1.
// (The former "+1" pad, 10 words per row, gave a 4-way conflict in the stride-16 round: 16 * 10 words = 0 mod 32.)
// The swizzle term sw2() is XOR-linear, and a round addresses rows row0 | mm (mm = slot << S0, a compile-time constant after
// unrolling, disjoint from row0's bits), so swz(row0 | mm) = ((row0 ^ sw2(row0)) ^ x) + (mm & ~3) with x = (mm & 3) ^ sw2(mm) a
// compile-time constant in 0..3: four base addresses per item, every access a base + immediate offset.
__host__ __device__ constexpr u32 sw2(u32 row) { return ((row >> 2) ^ (row >> 4) ^ (row >> 6) ^ (row >> 8)) & 3u; }
__device__ __forceinline__ u32 swz(u32 row) { return row ^ sw2(row); }
// element index of tile row (row0 | mm), column q
__device__ __forceinline__ u32 tile_at(u32 row0, u32 mm, u32 q) {
    const u32 base = row0 ^ sw2(row0);
    const u32 x = (mm & 3u) ^ sw2(mm);
    return ((base ^ x) * kXt + q) + (mm & ~3u) * kXt;
}
constexpr int kMaxLogT = 10;      // tile points
constexpr int kTwLog = 10;        // w_1024 table, full period

using gl::gf::add;
using gl::gf::mul;
using gl::gf::sub;

// two_adic_generator(k) = 2^root_exp(k) for k <= 6 (checked against the host field when a context starts, and in tests);
// inverse = 2^(192 - e). two_adic_generator(7) is not a power of two.
__host__ __device__ constexpr int root_exp(int logr, bool inv) {
    int e = logr == 1 ? 96 : logr == 2 ? 48 : logr == 3 ? 120 : logr == 4 ? 156 : logr == 5 ? 78 : logr == 6 ? 39 : 0;
    return inv ? (192 - e) % 192 : e;
}

// (u - x) * 2^e, e in [0, 192) known at compile time after unrolling
__device__ __forceinline__ u64 sub_mul_pow2(u64 u, u64 x, int e) {
    if (e == 0) return sub(u, x);
    if (e == 96) return sub(x, u);
    if (e < 96) return gl::gf::mul_pow2(sub(u, x), e);
    return gl::gf::mul_pow2(sub(x, u), e - 96);
}
// x * 2^e for canonical x, e in [0, 192) known at compile time after unrolling: 2^96 = -1, and -x = p - x costs no reduction
// because mul_pow2 takes any u64
__device__ __forceinline__ u64 mul_pow2_any(u64 x, int e) {
    if (e == 0) return x;
    if (e == 96) return sub(0, x);
    if (e < 96) return gl::gf::mul_pow2(x, e);
    return gl::gf::mul_pow2(GLD_P - x, e - 96);
}

// size-2^RB DFT in registers, natural order in, bit-reversed order out (decimation in frequency)
template <int RB, bool INV>
__device__ __forceinline__ void dif_regs(u64 (&v)[1 << RB]) {
    constexpr int R = 1 << RB;
#pragma unroll
    for (int s = 0; s < RB; s++) {
        const int half = R >> (s + 1);
        const int lg = RB - s;
#pragma unroll
        for (int blk = 0; blk < R; blk += 2 * half) {
#pragma unroll
            for (int el = 0; el < half; el++) {
                const int i = blk + el, j = i + half;
                const int e = (root_exp(lg, INV) * el) % 192;
                u64 u = v[i], x = v[j];
                v[i] = add(u, x);
                v[j] = sub_mul_pow2(u, x, e);
            }
        }
    }
}
// bit-reversed order in, natural order out (decimation in time)
template <int RB, bool INV>
__device__ __forceinline__ void dit_regs(u64 (&v)[1 << RB]) {
    constexpr int R = 1 << RB;
#pragma unroll
    for (int s = 0; s < RB; s++) {
        const int half = 1 << s;
        const int lg = s + 1;
#pragma unroll
        for (int blk = 0; blk < R; blk += 2 * half) {
#pragma unroll
            for (int el = 0; el < half; el++) {
                const int i = blk + el, j = i + half;
                const int e = (root_exp(lg, INV) * el) % 192;
                u64 u = v[i], x = v[j];
                if (e == 0) {
                    v[i] = add(u, x);
                    v[j] = sub(u, x);
                } else if (e == 96) {
                    v[i] = sub(u, x);
                    v[j] = add(u, x);
                } else if (e < 96) {
                    u64 y = gl::gf::mul_pow2(x, e);
                    v[i] = add(u, y);
                    v[j] = sub(u, y);
                } else {
                    u64 y = gl::gf::mul_pow2(x, e - 96);
                    v[i] = sub(u, y);
                    v[j] = add(u, y);
                }
            }
        }
    }
}

__host__ __device__ constexpr int rev_small(int x, int bits) {
    int r = 0;
    for (int i = 0; i < bits; i++) r |= ((x >> i) & 1) << (bits - 1 - i);
    return r;
}

// Round sizes of a tb-bit DIF tile from the top bits down: 4, 4, rest. A DIT tile runs the same rounds in mirror order from
// the low bits up (rest, 4, 4), so both run the same (size, bit offset) rounds with the same twiddles -- except at tb = 7,
// where DIT keeps 4, 3: its mirror 3, 4 would pay the general (order-128) twiddles on 15 of 16 elements instead of 7 of 8.
__host__ __device__ constexpr int round_bits(int tb, int k) {
    int r1 = tb < 4 ? tb : 4, rem = tb - r1;
    int r2 = rem < 4 ? rem : 4;
    return k == 0 ? r1 : k == 1 ? r2 : rem - r2;
}

// One round of RB bits at bit offset S0 of a TB-bit tile. Slot m of item (blk, off) is tile row
// (blk << (S0 + RB)) + off + (m << S0). DIF: DFT then slot m *= w^{off * rev(m)}; DIT: the mirror image.
// w = w_{2^(S0+RB)}: when S0 + RB <= 6 it is a power of two (the radix-16 round over bits [2, 6) of a 10-bit tile, [1, 5) of a
// 9-bit one), and the twiddles are shifts by compile-time amounts, one unrolled body per value of off (off < 2^S0 <= 4). off
// is taken from the HIGH bits of the item index so that it is warp-uniform (8 thread rows of a warp share it whenever a value
// of off has >= 8 items): 256 threads, 64 items, off = trow >> 4. The half-warp's 4 rows then differ in two adjacent row bits
// above bit 1 (bits 6-7 at TB = 10, 5-6 at TB = 9), which sw2() maps one-to-one onto the bank group: no conflict
// (tools/smem_banks.py counts every round).
// ld(row0, mm) / st(row0, mm, value) move the element of tile row row0 | mm of this thread's column (registers <-> global or
// shared memory); mm = m << S0 is a compile-time constant after unrolling.
// post (the LAST round only): table of the pass's output multipliers (inter-pass twiddles), indexed by tile row, or null.
// Its loads are issued for the whole item BEFORE the butterflies (radix <= 4: 8 registers) or right after them, never between
// the stores: written as "load, multiply, store" per element the compiler keeps that order (the stores may alias the table as
// far as it knows) and every element waits a full L2 round trip on its own -- 22 % of all stall samples of the fused LDE
// kernel (profiles/ncu_lde_mid_r2_v1.txt).
template <int TB, int RB, int S0, bool INV, bool DIT, class Ld, class St>
__device__ __forceinline__ void tile_round(const u64* __restrict__ tw, u32 trow, u32 nrows_thr, Ld ld, St st, const u64* __restrict__ post_tab = nullptr) {
    constexpr int R = 1 << RB;
    constexpr u32 items = 1u << (TB - RB);
    constexpr bool kEarlyPost = R <= 4;
    constexpr int kBlkBits = TB - RB - S0;
    constexpr bool kShiftTw = S0 > 0 && S0 + RB <= 6;
    auto twiddle = [&](u64(&v)[R], u32 off) {
        if constexpr (kShiftTw) {
#pragma unroll
            for (int o = 1; o < (1 << S0); o++) {
                if (off == (u32)o) {
#pragma unroll
                    for (int m = 1; m < R; m++) v[m] = mul_pow2_any(v[m], (root_exp(S0 + RB, INV) * o * rev_small(m, RB)) % 192);
                }
            }
        } else if constexpr (S0 > 0) {
#pragma unroll
            for (int m = 1; m < R; m++) v[m] = mul(v[m], __ldg(tw + ((off * (u32)rev_small(m, RB)) << (kTwLog - S0 - RB))));
        }
    };
    for (u32 g = trow; g < items; g += nrows_thr) {
        const u32 off = S0 > 0 ? g >> kBlkBits : 0u, blk = S0 > 0 ? g & ((1u << kBlkBits) - 1) : g;
        const u32 row0 = (blk << (S0 + RB)) + off;
        u64 v[R], pt[R];
        if (kEarlyPost && post_tab) {
#pragma unroll
            for (int m = 0; m < R; m++) pt[m] = __ldg(post_tab + row0 + ((u32)m << S0));
        }
#pragma unroll
        for (int m = 0; m < R; m++) v[m] = ld(row0, (u32)m << S0);
        if (DIT) {
            twiddle(v, off);
            dit_regs<RB, INV>(v);
        } else {
            dif_regs<RB, INV>(v);
            twiddle(v, off);
        }
        if (post_tab) {
            if (!kEarlyPost) {
#pragma unroll
                for (int m = 0; m < R; m++) pt[m] = __ldg(post_tab + row0 + ((u32)m << S0));
            }
#pragma unroll
            for (int m = 0; m < R; m++) v[m] = mul(v[m], pt[m]);
        }
#pragma unroll
        for (int m = 0; m < R; m++) st(row0, (u32)m << S0, v[m]);
    }
}

// All rounds of a TB-bit tile for this thread's column q. gld(row) reads the input element of tile row `row`,
// gst(row, v) consumes the output element. DIF: natural rows in, bit-reversed rows out. DIT: the converse.
template <int TB, bool INV, bool DIT, class GLd, class GSt>
__device__ __forceinline__ void tile_pass(u64* tile, const u64* __restrict__ tw, u32 q, u32 trow, u32 nrows_thr, GLd gld, GSt gst,
                                          const u64* __restrict__ post = nullptr) {
    constexpr int B0 = round_bits(TB, 0), B1 = round_bits(TB, 1), B2 = round_bits(TB, 2);
    auto sld = [&](u32 row0, u32 mm) { return tile[tile_at(row0, mm, q)]; };
    auto sst = [&](u32 row0, u32 mm, u64 v) { tile[tile_at(row0, mm, q)] = v; };
    if constexpr (!DIT) {
        // round 0 works on the top bits
        if constexpr (B1 == 0) {
            tile_round<TB, B0, TB - B0, INV, false>(tw, trow, nrows_thr, gld, gst, post);
        } else if constexpr (B2 == 0) {
            tile_round<TB, B0, TB - B0, INV, false>(tw, trow, nrows_thr, gld, sst);
            __syncthreads();
            tile_round<TB, B1, 0, INV, false>(tw, trow, nrows_thr, sld, gst, post);
        } else {
            tile_round<TB, B0, TB - B0, INV, false>(tw, trow, nrows_thr, gld, sst);
            __syncthreads();
            tile_round<TB, B1, B2, INV, false>(tw, trow, nrows_thr, sld, sst);
            __syncthreads();
            tile_round<TB, B2, 0, INV, false>(tw, trow, nrows_thr, sld, gst, post);
        }
    } else {
        // the DIF rounds in mirror order: round 0 works on the low bits
        if constexpr (B1 == 0) {
            tile_round<TB, B0, 0, INV, true>(tw, trow, nrows_thr, gld, gst, post);
        } else if constexpr (B2 == 0) {
            constexpr int D0 = TB == 7 ? B0 : B1, D1 = TB - D0;
            tile_round<TB, D0, 0, INV, true>(tw, trow, nrows_thr, gld, sst);
            __syncthreads();
            tile_round<TB, D1, D0, INV, true>(tw, trow, nrows_thr, sld, gst, post);
        } else {
            tile_round<TB, B2, 0, INV, true>(tw, trow, nrows_thr, gld, sst);
            __syncthreads();
            tile_round<TB, B1, B2, INV, true>(tw, trow, nrows_thr, sld, sst);
            __syncthreads();
            tile_round<TB, B0, B1 + B2, INV, true>(tw, trow, nrows_thr, sld, gst, post);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Strided decimation-in-frequency pass.
// Element (a, j, x) of the pass lives at ((a*T + j)*I + x); the pass transforms j for every (a, x),
// then multiplies the output at tile row r (frequency k1 = rev(r)) by w_M^{(x / w) * k1}, M = T*I/w.
// ------------------------------------------------------------------------------------------------
struct StridedParams {
    const u64* src;
    u64* dst;
    const u64* tw;    // w_1024^{+-i}, i < 1024
    const u64* twp;   // inter-pass twiddles [b][r] = w_M^{+-b * rev(r)}, or null
    u64 I;            // inner elements per point: S * w
    u64 a_total;      // number of (independent) outer blocks
    u32 w;
};

template <int TB, bool INV>
__global__ void __launch_bounds__(64 * kXt, 1024 / (64 * kXt)) k_ntt_strided(StridedParams p) {
    extern __shared__ u64 smem[];
    constexpr u32 T = 1u << TB;
    const u32 q = threadIdx.x & (kXt - 1), trow = threadIdx.x >> kLogXt, nrows_thr = blockDim.x >> kLogXt;
    // this thread's column: element offset of tile row 0, validity, and the row index b of the inter-pass twiddle
    // Virtual column v enumerates (outer block a, inner index x): tiles take kXt consecutive virtual columns, so lanes
    // are idle only in the very last tile even when the row length is not a multiple of kXt.
    const u64 v = (u64)blockIdx.x * kXt + q;
    const bool valid = v < p.a_total * p.I;
    const u64 a = valid ? v / p.I : 0, x = valid ? v % p.I : 0;
    const u64 col = a * T * p.I + x;
    const u32 b = (u32)(x / p.w);
    const u64* __restrict__ src = p.src + col;
    u64* __restrict__ dst = p.dst + col;
    const u64 I = p.I;
    const u64* __restrict__ twp = p.twp ? p.twp + (size_t)b * T : nullptr;
    auto gld = [&](u32 row0, u32 mm) -> u64 { return valid ? src[(u64)(row0 + mm) * I] : 0ull; };
    auto gst = [&](u32 row0, u32 mm, u64 v) {
        if (valid) dst[(u64)(row0 + mm) * I] = v;
    };
    tile_pass<TB, INV, false>(smem, p.tw, q, trow, nrows_thr, gld, gst, twp);
}

// ------------------------------------------------------------------------------------------------
// Block pass: first pass of the coset evaluations from bit-reversed coefficients.
// src position p = (blk, t): coefficient j = rev_T(t) * S + rev_{L-tb}(blk). For low index b, the tile
// reads block rev(b), scales by scale[beta](j), runs a DIT tile (row s = frequency k1 = s), multiplies
// by w_n^{b*k1} and stores row s at destination row rev_T(s) * S + b of output block beta.
// ------------------------------------------------------------------------------------------------
struct BlockParams {
    const u64* src;
    u64* dst;
    const u64* tw;      // w_1024^i
    const u64* scale;   // [beta][b][t] = (shift_beta)^{rev_T(t)*S + b} / n
    const u64* twb;     // [b][s] = w_n^{b*s}, or null when S == 1
    u64 S;              // n / T
    u64 out_block_elems;  // n * w
    u32 log_n, w;
};

template <int TB>
__global__ void __launch_bounds__(64 * kXt, 1024 / (64 * kXt)) k_ntt_block(BlockParams p) {
    extern __shared__ u64 smem[];
    constexpr u32 T = 1u << TB;
    const u32 q = threadIdx.x & (kXt - 1), trow = threadIdx.x >> kLogXt, nrows_thr = blockDim.x >> kLogXt;
    const u32 hi_bits = p.log_n - TB;
    const u32 w = p.w;
    // virtual column v = b * w + c over the S low indices b and the w matrix columns c
    const u64 v = (u64)blockIdx.x * kXt + q;
    const bool valid = v < p.S * w;
    const u64 b = valid ? v / w : 0;
    const u32 c = valid ? (u32)(v % w) : 0;
    const u64 blk = gl::rev_bits((u32)b, hi_bits);
    const u64* __restrict__ src = p.src + blk * T * w + c;
    const u64* __restrict__ sc = p.scale + ((size_t)blockIdx.y * p.S + b) * T;
    const u64* __restrict__ twb = p.twb ? p.twb + (size_t)b * T : nullptr;
    u64* __restrict__ dst = p.dst + (u64)blockIdx.y * p.out_block_elems + b * w + c;
    const u64 dstride = p.S * w;
    auto gld = [&](u32 t0, u32 mm) -> u64 { const u32 t = t0 + mm; return valid ? mul(src[(u64)t * w], __ldg(sc + t)) : 0ull; };
    auto gst = [&](u32 s0, u32 mm, u64 v) {
        if (valid) dst[(u64)gl::rev_bits(s0 + mm, TB) * dstride] = v;
    };
    tile_pass<TB, false, true>(smem, p.tw, q, trow, nrows_thr, gld, gst, twb);
}

// ------------------------------------------------------------------------------------------------
// Fused middle pass of the coset LDE: LAST inverse pass + FIRST forward pass of every coset in one kernel.
// The last inverse pass (bits [0, tb), contiguous blocks of T rows) leaves tile position t holding the coefficient
// j = rev_T(t) * S + rev(blk) -- exactly the tile the block pass of each coset starts from. So a CTA runs the inverse
// DIF tile once, keeps the coefficients in a shared-memory tile A, and then for every coset beta scales them by
// shift_beta^j / n, runs the DIT tile in a second (work) tile and scatters the row segments to output block beta.
// The coefficients cross HBM never: one read of n*w for all B cosets instead of one write + B reads, and the
// unnormalised inverse's last pass costs no launch of its own.
// ------------------------------------------------------------------------------------------------
struct MidParams {
    const u64* src;     // evaluations (log_n <= tb) or the output of the earlier inverse passes; natural rows per T-block
    u64* dst;
    const u64* tw_inv;  // w_1024^{-i}
    const u64* tw_fwd;  // w_1024^{i}
    const u64* scale;   // [beta][b][t] = (shift_beta)^{rev_T(t)*S + b} / n
    const u64* twb;     // [b][s] = w_n^{b*s}, or null when S == 1
    u64 S;              // n / T
    u64 out_block_elems;  // n * w
    u32 log_n, w, n_cosets;
};

template <int TB>
__global__ void __launch_bounds__(64 * kXt, 3) k_lde_mid(MidParams p) {
    extern __shared__ u64 smem[];
    constexpr u32 T = 1u << TB;
    u64* A = smem;                 // coefficients of this tile (canonical), read by every coset
    u64* W = smem + T * kXt;       // work tile of the forward rounds (unused when the tile is a single round)
    const u32 q = threadIdx.x & (kXt - 1), trow = threadIdx.x >> kLogXt, nrows_thr = blockDim.x >> kLogXt;
    const u32 hi_bits = p.log_n - TB;
    const u32 w = p.w;
    const u64 v = (u64)blockIdx.x * kXt + q;   // virtual column b * w + c
    const bool valid = v < p.S * w;
    const u64 b = valid ? v / w : 0;
    const u32 c = valid ? (u32)(v % w) : 0;
    const u64 blk = gl::rev_bits((u32)b, hi_bits);
    const u64* __restrict__ src = p.src + blk * T * w + c;
    // ---- inverse DIF tile: natural rows in, coefficient rev_T(t) at tile row t, left in A ----
    {
        auto gld = [&](u32 row0, u32 mm) -> u64 { return valid ? src[(u64)(row0 + mm) * w] : 0ull; };
        auto ast = [&](u32 t0, u32 mm, u64 x) { A[tile_at(t0, mm, q)] = x; };
        tile_pass<TB, true, false>(A, p.tw_inv, q, trow, nrows_thr, gld, ast);
    }
    __syncthreads();
    const u64* __restrict__ twb = p.twb ? p.twb + (size_t)b * T : nullptr;
    const u64 dstride = p.S * w;
    for (u32 beta = 0; beta < p.n_cosets; beta++) {
        const u64* __restrict__ sc = p.scale + ((size_t)beta * p.S + b) * T;
        u64* __restrict__ dst = p.dst + (u64)beta * p.out_block_elems + b * w + c;
        auto ald = [&](u32 t0, u32 mm) -> u64 { return mul(A[tile_at(t0, mm, q)], __ldg(sc + t0 + mm)); };
        auto gst = [&](u32 s0, u32 mm, u64 x) {
            if (valid) dst[(u64)gl::rev_bits(s0 + mm, TB) * dstride] = x;
        };
        tile_pass<TB, false, true>(W, p.tw_fwd, q, trow, nrows_thr, ald, gst, twb);
        __syncthreads();   // the next coset's first round overwrites W
    }
}

// dst[beta][j][c] = src[j][c] * tab[beta](j)
__global__ void k_scale_rows(const u64* src, u64* dst, u64 n, u64 w, const gl::PowTable* tabs, u32 nb) {
    u64 total = n * w;
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (u64)gridDim.x * blockDim.x) {
        u64 j = e / w;
        u64 v = src[e];
        for (u32 beta = 0; beta < nb; beta++) dst[(u64)beta * total + e] = gl::mul(v, gl::pow_lookup(tabs[beta], j));
    }
}

// dst[r][c] = src[rev(r)][c] * scalar
__global__ void k_bitrev_rows_scale(const u64* src, u64* dst, u64 n, u64 w, u32 log_n, u64 scalar) {
    u64 total = n * w;
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (u64)gridDim.x * blockDim.x) {
        u64 r = e / w, c = e % w;
        u64 v = src[(u64)gl::rev_bits((u32)r, log_n) * w + c];
        dst[e] = scalar == 1 ? v : gl::mul(v, scalar);
    }
}

// ---- table builders ----------------------------------------------------------------------------------
// out[b * T + r] = g^{b * rev_tb(r)}
__global__ void k_fill_twp(u64* out, u64 total, u32 tb, gl::PowTable g) {
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (u64)gridDim.x * blockDim.x) {
        u64 b = e >> tb;
        u32 r = (u32)(e & ((1u << tb) - 1));
        out[e] = gl::pow_lookup(g, b * gl::rev_bits(r, tb));
    }
}
// out[b * T + s] = g^{b * s}
__global__ void k_fill_twb(u64* out, u64 total, u32 tb, gl::PowTable g) {
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (u64)gridDim.x * blockDim.x) {
        u64 b = e >> tb;
        u32 s = (u32)(e & ((1u << tb) - 1));
        out[e] = gl::pow_lookup(g, b * s);
    }
}
// out[(beta * S + b) * T + t] = tab[beta](rev_tb(t) * S + b)
__global__ void k_fill_scale(u64* out, u64 n, u32 tb, u64 S, const gl::PowTable* tabs, u32 nb) {
    u64 total = n * nb;
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (u64)gridDim.x * blockDim.x) {
        u32 t = (u32)(e & ((1u << tb) - 1));
        u64 rest = e >> tb;
        u64 b = rest % S, beta = rest / S;
        out[e] = gl::pow_lookup(tabs[beta], (u64)gl::rev_bits(t, tb) * S + b);
    }
}

// ------------------------------------------------------------------------------------------------
// Host drivers
// ------------------------------------------------------------------------------------------------
static std::vector<u32> plan_passes(u32 log_n) {
    std::vector<u32> tb;
    if (log_n == 0) return tb;
    u32 np = (log_n + kMaxLogT - 1) / kMaxLogT;
    u32 base = log_n / np, rem = log_n % np;
    for (u32 i = 0; i < np; i++) tb.push_back(base + (i < rem ? 1 : 0));
    return tb;
}

static size_t tile_smem(u32 log_t) { return log_t <= 4 ? 0 : (size_t)(1u << log_t) * kXt * sizeof(u64); }
static u32 tile_threads(u32 log_t) {
    u32 rows = log_t >= 4 ? (1u << (log_t - 4)) : 1u;  // one thread row per radix-16 item
    u32 t = rows * kXt;
    if (t < 32) t = 32;
    if (t > 64 * kXt) t = 64 * kXt;
    return t;
}

template <int TB>
static void launch_strided_tb(const StridedParams& p, bool inverse, u64 blocks, cudaStream_t st) {
    if (inverse) {
        ensure_max_smem(k_ntt_strided<TB, true>, (int)tile_smem(kMaxLogT));
        k_ntt_strided<TB, true><<<(unsigned)blocks, tile_threads(TB), tile_smem(TB), st>>>(p);
    } else {
        ensure_max_smem(k_ntt_strided<TB, false>, (int)tile_smem(kMaxLogT));
        k_ntt_strided<TB, false><<<(unsigned)blocks, tile_threads(TB), tile_smem(TB), st>>>(p);
    }
}
template <int TB>
static void launch_block_tb(const BlockParams& p, dim3 grid, cudaStream_t st) {
    ensure_max_smem(k_ntt_block<TB>, (int)tile_smem(kMaxLogT));
    k_ntt_block<TB><<<grid, tile_threads(TB), tile_smem(TB), st>>>(p);
}

static size_t mid_smem(u32 log_t) { return (size_t)(1u << log_t) * kXt * sizeof(u64) * (log_t <= 4 ? 1 : 2); }
template <int TB>
static void launch_mid_tb(const MidParams& p, unsigned blocks, cudaStream_t st) {
    ensure_max_smem(k_lde_mid<TB>, (int)mid_smem(kMaxLogT));
    k_lde_mid<TB><<<blocks, tile_threads(TB), mid_smem(TB), st>>>(p);
}

#define MSG_TB_SWITCH(tb, CALL)                               \
    switch (tb) {                                             \
        case 1: { constexpr int TBV = 1; CALL; } break;       \
        case 2: { constexpr int TBV = 2; CALL; } break;       \
        case 3: { constexpr int TBV = 3; CALL; } break;       \
        case 4: { constexpr int TBV = 4; CALL; } break;       \
        case 5: { constexpr int TBV = 5; CALL; } break;       \
        case 6: { constexpr int TBV = 6; CALL; } break;       \
        case 7: { constexpr int TBV = 7; CALL; } break;       \
        case 8: { constexpr int TBV = 8; CALL; } break;       \
        case 9: { constexpr int TBV = 9; CALL; } break;       \
        case 10: { constexpr int TBV = 10; CALL; } break;     \
        default: throw Error(-3, "ntt: bad tile size");       \
    }

// inter-pass twiddle table of a DIF pass: [b][r] = w_{2^log_big}^{+-b * rev_tb(r)}, b < 2^(log_big - tb)
static const u64* twp_table(Ctx& c, u32 log_big, u32 tb, bool inverse) {
    auto key = std::make_tuple(0u, log_big, tb, (u64)inverse);
    auto it = c.ntt_tables.find(key);
    if (it != c.ntt_tables.end()) return it->second;
    msh::Fp g = msh::two_adic_generator(log_big);
    if (inverse) g = g.inverse();
    gl::PowTable tab = c.pow_table(g.v, 1, log_big).view();
    u64 total = 1ull << log_big;
    u64* d;
    MSG_CUDA(cudaMalloc(&d, total * 8));
    c.owned.push_back(d);
    k_fill_twp<<<(unsigned)std::min<u64>((total + 255) / 256, (u64)c.sm_count * 16), 256, 0, c.stream>>>(d, total, tb, tab);
    MSG_CUDA(cudaGetLastError());
    c.ntt_tables[key] = d;
    return d;
}
// output twiddle table of the block pass: [b][s] = w_n^{b * s}
static const u64* twb_table(Ctx& c, u32 log_n, u32 tb) {
    auto key = std::make_tuple(1u, log_n, tb, (u64)0);
    auto it = c.ntt_tables.find(key);
    if (it != c.ntt_tables.end()) return it->second;
    gl::PowTable tab = c.pow_table(msh::two_adic_generator(log_n).v, 1, log_n).view();
    u64 total = 1ull << log_n;
    u64* d;
    MSG_CUDA(cudaMalloc(&d, total * 8));
    c.owned.push_back(d);
    k_fill_twb<<<(unsigned)std::min<u64>((total + 255) / 256, (u64)c.sm_count * 16), 256, 0, c.stream>>>(d, total, tb, tab);
    MSG_CUDA(cudaGetLastError());
    c.ntt_tables[key] = d;
    return d;
}
// coset scales of the block pass: [beta][b][t] = (shift * w_{nB}^{rev(beta)})^{rev_tb(t) * S + b} / n
static const u64* scale_table(Ctx& c, u32 log_n, u32 tb, u32 added_bits, u64 shift) {
    auto key = std::make_tuple(2u + (added_bits << 8), log_n, tb, shift);
    auto it = c.ntt_tables.find(key);
    if (it != c.ntt_tables.end()) return it->second;
    const gl::PowTable* tabs = c.coset_tables(log_n, added_bits, shift);
    u64 n = 1ull << log_n, total = n << added_bits;
    u64* d;
    MSG_CUDA(cudaMalloc(&d, total * 8));
    c.owned.push_back(d);
    k_fill_scale<<<(unsigned)std::min<u64>((total + 255) / 256, (u64)c.sm_count * 16), 256, 0, c.stream>>>(d, n, tb, n >> tb, tabs,
                                                                                                         1u << added_bits);
    MSG_CUDA(cudaGetLastError());
    c.ntt_tables[key] = d;
    return d;
}

// One DIF pass over bits [lo_bit, lo_bit + tb) of a size-2^log_m transform, for `count` transforms
// stored back to back (count * 2^log_m rows in total).
static void launch_strided(Ctx& c, const u64* src, u64* dst, u32 log_m, u64 count, u64 w, u32 lo_bit, u32 tb, bool inverse) {
    StridedParams p{};
    p.src = src;
    p.dst = dst;
    p.tw = c.tw_full[inverse ? 1 : 0];
    p.w = (u32)w;
    u64 S = 1ull << lo_bit;
    p.I = S * w;
    p.a_total = count << (log_m - lo_bit - tb);
    p.twp = lo_bit > 0 ? twp_table(c, lo_bit + tb, tb, inverse) : nullptr;
    u64 blocks = (p.a_total * p.I + kXt - 1) / kXt;
    MSG_REQUIRE(blocks < (1ull << 31), "ntt: grid too large");
    {
        KLaunch kl(c, "k_ntt_strided");
        MSG_TB_SWITCH(tb, launch_strided_tb<TBV>(p, inverse, blocks, c.stream));
    }
    MSG_CUDA(cudaGetLastError());
}

void ntt_dft_bitrev(Ctx& c, const u64* src, u64* dst, u64 n, u64 w, bool inverse, u64 batch) {
    MSG_REQUIRE(is_pow2(n), "ntt: height must be a power of two");
    if (w == 0 || batch == 0) return;
    u32 log_n = ilog2(n);
    MSG_REQUIRE(log_n <= msh::GL_TWO_ADICITY, "ntt: height exceeds the two-adicity of the field");
    auto plan = plan_passes(log_n);
    if (plan.empty()) {
        if (src != dst) MSG_CUDA(cudaMemcpyAsync(dst, src, batch * n * w * 8, cudaMemcpyDeviceToDevice, c.stream));
        return;
    }
    u32 hi = log_n;
    const u64* cur = src;
    for (u32 tb : plan) {
        launch_strided(c, cur, dst, log_n, batch, w, hi - tb, tb, inverse);
        cur = dst;
        hi -= tb;
    }
}

void ntt_coset_lde(Ctx& c, const u64* src, u64* dst, u64* tmp, u64 n, u64 w, u32 added_bits, u64 shift) {
    MSG_REQUIRE(is_pow2(n), "lde: height must be a power of two");
    if (w == 0) return;
    u32 log_n = ilog2(n);
    MSG_REQUIRE(log_n + added_bits <= msh::GL_TWO_ADICITY, "lde: extended height exceeds the two-adicity of the field");
    if (log_n == 0) {  // constant polynomials: every coset evaluation is the value itself
        for (u64 beta = 0; beta < (1ull << added_bits); beta++)
            MSG_CUDA(cudaMemcpyAsync(dst + beta * w, src, w * 8, cudaMemcpyDeviceToDevice, c.stream));
        return;
    }
    auto plan = plan_passes(log_n);
    u32 tb = plan.back();
    static const bool fused = !(getenv("MSGPU_LDE_UNFUSED") && getenv("MSGPU_LDE_UNFUSED")[0] == '1');
    if (fused) {
        // 1. inverse passes over the upper bits (unnormalised, natural -> bit-reversed in place); the last one is fused below
        const u64* cur = src;
        u32 hi = log_n;
        for (size_t i = 0; i + 1 < plan.size(); i++) {
            launch_strided(c, cur, tmp, log_n, 1, w, hi - plan[i], plan[i], true);
            cur = tmp;
            hi -= plan[i];
        }
        // 2. last inverse pass + first forward pass of every coset
        MidParams p{};
        p.src = cur;
        p.dst = dst;
        p.tw_inv = c.tw_full[1];
        p.tw_fwd = c.tw_full[0];
        p.scale = scale_table(c, log_n, tb, added_bits, shift);
        p.log_n = log_n;
        p.w = (u32)w;
        p.n_cosets = 1u << added_bits;
        p.S = n >> tb;
        p.out_block_elems = n * w;
        p.twb = p.S > 1 ? twb_table(c, log_n, tb) : nullptr;
        u64 blocks = (p.S * w + kXt - 1) / kXt;
        MSG_REQUIRE(blocks < (1ull << 31), "lde: grid too large");
        {
            KLaunch kl(c, "k_lde_mid");
            MSG_TB_SWITCH(tb, launch_mid_tb<TBV>(p, (unsigned)blocks, c.stream));
        }
        MSG_CUDA(cudaGetLastError());
    } else {
    // 1. inverse transform (unnormalised): coefficients in bit-reversed order
    ntt_dft_bitrev(c, src, tmp, n, w, true);
    // 2. first forward pass per coset from the bit-reversed coefficients
    BlockParams p{};
    p.src = tmp;
    p.dst = dst;
    p.tw = c.tw_full[0];
    p.scale = scale_table(c, log_n, tb, added_bits, shift);
    p.log_n = log_n;
    p.w = (u32)w;
    p.S = n >> tb;
    p.out_block_elems = n * w;
    p.twb = p.S > 1 ? twb_table(c, log_n, tb) : nullptr;
    u64 blocks = (p.S * w + kXt - 1) / kXt;
    MSG_REQUIRE(blocks < (1ull << 31), "lde: grid too large");
    dim3 grid((unsigned)blocks, 1u << added_bits);
    {
        KLaunch kl(c, "k_ntt_block");
        MSG_TB_SWITCH(tb, launch_block_tb<TBV>(p, grid, c.stream));
    }
    MSG_CUDA(cudaGetLastError());
    }
    // 3. remaining forward passes: every block rev_T(k1) of S rows is an independent size-S DFT
    u32 log_s = log_n - tb;
    if (log_s > 0) {
        auto rest = plan_passes(log_s);
        u32 hi = log_s;
        u64 count = (n >> log_s) << added_bits;
        for (u32 t2 : rest) {
            launch_strided(c, dst, dst, log_s, count, w, hi - t2, t2, false);
            hi -= t2;
        }
    }
}

void ntt_lde_from_coeffs(Ctx& c, const u64* src, u64* dst, u64 n, u64 w, u32 added_bits) {
    MSG_REQUIRE(is_pow2(n), "lde: height must be a power of two");
    if (w == 0) return;
    u32 log_n = ilog2(n);
    MSG_REQUIRE(log_n + added_bits <= msh::GL_TWO_ADICITY, "lde: extended height exceeds the two-adicity of the field");
    const gl::PowTable* tabs = c.lde_coeff_tables(log_n, added_bits);
    u64 total = n * w;
    unsigned blocks = (unsigned)std::min<u64>((total + 255) / 256, (u64)c.sm_count * 16);
    {
        KLaunch kl(c, "k_scale_rows");
        k_scale_rows<<<blocks, 256, 0, c.stream>>>(src, dst, n, w, tabs, 1u << added_bits);
    }
    MSG_CUDA(cudaGetLastError());
    ntt_dft_bitrev(c, dst, dst, n, w, false, 1ull << added_bits);
}

void ntt_bit_reverse_rows(Ctx& c, const u64* src, u64* dst, u64 n, u64 w) {
    if (n * w == 0) return;
    u64 total = n * w;
    unsigned blocks = (unsigned)std::min<u64>((total + 255) / 256, (u64)c.sm_count * 16);
    {
        KLaunch kl(c, "k_bitrev_rows_scale");
        k_bitrev_rows_scale<<<blocks, 256, 0, c.stream>>>(src, dst, n, w, ilog2(n), 1);
    }
    MSG_CUDA(cudaGetLastError());
}

void ntt_idft_natural(Ctx& c, const u64* src, u64* dst, u64* tmp, u64 n, u64 w) {
    if (n * w == 0) return;
    ntt_dft_bitrev(c, src, tmp, n, w, true);
    u64 total = n * w;
    unsigned blocks = (unsigned)std::min<u64>((total + 255) / 256, (u64)c.sm_count * 16);
    {
        KLaunch kl(c, "k_bitrev_rows_scale");
        k_bitrev_rows_scale<<<blocks, 256, 0, c.stream>>>(tmp, dst, n, w, ilog2(n), msh::Fp((msh::u64)n).inverse().v);
    }
    MSG_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------
// Tables
// ------------------------------------------------------------------------------------------------
DevPow Ctx::pow_table(u64 g, u64 cst, u32 bits) {
    auto key = std::make_tuple(g, cst, bits);
    auto it = pow_cache.find(key);
    if (it != pow_cache.end()) return it->second;
    DevPow t;
    t.h1 = (bits + 1) / 2;
    size_t nlo = (size_t)1 << t.h1, nhi = (size_t)1 << (bits - t.h1);
    std::vector<u64> lo(nlo), hi(nhi);
    msh::Fp G(g), acc(cst);
    for (size_t i = 0; i < nlo; i++) { lo[i] = acc.v; acc *= G; }
    msh::Fp Gh = G.exp_power_of_2(t.h1);
    acc = msh::Fp::one();
    for (size_t i = 0; i < nhi; i++) { hi[i] = acc.v; acc *= Gh; }
    MSG_CUDA(cudaMalloc(&t.lo, nlo * 8));
    MSG_CUDA(cudaMalloc(&t.hi, nhi * 8));
    owned.push_back(t.lo);
    owned.push_back(t.hi);
    MSG_CUDA(cudaMemcpyAsync(t.lo, lo.data(), nlo * 8, cudaMemcpyHostToDevice, stream));
    MSG_CUDA(cudaMemcpyAsync(t.hi, hi.data(), nhi * 8, cudaMemcpyHostToDevice, stream));
    MSG_CUDA(cudaStreamSynchronize(stream));  // the host vectors die here
    pow_cache[key] = t;
    return t;
}

static const gl::PowTable* upload_views(Ctx& c, const std::vector<gl::PowTable>& v) {
    gl::PowTable* d;
    MSG_CUDA(cudaMalloc(&d, v.size() * sizeof(gl::PowTable)));
    c.owned.push_back(d);
    MSG_CUDA(cudaMemcpyAsync(d, v.data(), v.size() * sizeof(gl::PowTable), cudaMemcpyHostToDevice, c.stream));
    MSG_CUDA(cudaStreamSynchronize(c.stream));
    return d;
}

// scale[beta](j) = (shift * w_{nB}^{rev_b(beta)})^j / n
const gl::PowTable* Ctx::coset_tables(u32 log_n, u32 added_bits, u64 shift) {
    auto key = std::make_tuple(log_n, added_bits, shift);
    auto it = coset_cache.find(key);
    if (it != coset_cache.end()) return it->second;
    u32 B = 1u << added_bits;
    msh::Fp wN = msh::two_adic_generator(log_n + added_bits);
    msh::Fp ninv = msh::Fp((msh::u64)1 << log_n).inverse();
    std::vector<gl::PowTable> views(B);
    for (u32 beta = 0; beta < B; beta++) {
        u32 s = (u32)msh::reverse_bits_len(beta, added_bits);
        msh::Fp g = msh::Fp(shift) * wN.pow(s);
        views[beta] = pow_table(g.v, ninv.v, log_n).view();
    }
    gl::PowTable* d = const_cast<gl::PowTable*>(upload_views(*this, views));
    coset_cache[key] = d;
    return d;
}

// tab[beta](j) = w_{nB}^{rev_b(beta) * j}
const gl::PowTable* Ctx::lde_coeff_tables(u32 log_n, u32 added_bits) {
    auto key = std::make_tuple(log_n, added_bits | 0x80000000u, (u64)0);
    auto it = coset_cache.find(key);
    if (it != coset_cache.end()) return it->second;
    u32 B = 1u << added_bits;
    msh::Fp wN = msh::two_adic_generator(log_n + added_bits);
    std::vector<gl::PowTable> views(B);
    for (u32 beta = 0; beta < B; beta++) {
        u32 s = (u32)msh::reverse_bits_len(beta, added_bits);
        views[beta] = pow_table(wN.pow(s).v, 1, log_n).view();
    }
    gl::PowTable* d = const_cast<gl::PowTable*>(upload_views(*this, views));
    coset_cache[key] = d;
    return d;
}

void ctx_init_tables(Ctx& c) {
    // the register DFTs hard-code two_adic_generator(k) = 2^root_exp(k): verify against the host field
    for (int k = 1; k <= 6; k++) {
        int e = root_exp(k, false);
        msh::Fp want = msh::two_adic_generator(k), got = msh::Fp(2).pow((msh::u64)e);
        if (want != got) throw Error(-3, "ntt: two-adic generator is not the expected power of two");
    }
    const size_t full = (size_t)1 << kTwLog;
    std::vector<u64> f(full), inv(full);
    msh::Fp w = msh::two_adic_generator(kTwLog), wi = w.inverse();
    msh::Fp a = msh::Fp::one(), b = msh::Fp::one();
    for (size_t i = 0; i < full; i++) { f[i] = a.v; inv[i] = b.v; a *= w; b *= wi; }
    for (int d = 0; d < 2; d++) {
        MSG_CUDA(cudaMalloc(&c.tw_full[d], full * 8));
        c.owned.push_back(c.tw_full[d]);
    }
    MSG_CUDA(cudaMemcpyAsync(c.tw_full[0], f.data(), full * 8, cudaMemcpyHostToDevice, c.stream));
    MSG_CUDA(cudaMemcpyAsync(c.tw_full[1], inv.data(), full * 8, cudaMemcpyHostToDevice, c.stream));
    MSG_CUDA(cudaStreamSynchronize(c.stream));
}

}  // namespace msg
