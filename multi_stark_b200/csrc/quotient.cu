// Constraint programs on the device: the quotient stage and the stage-2 (logUp) trace construction.
//
// Replaces, for one circuit, the reference's
//   quotient_values + quotient_values_inner      src/prover.rs:756-962
//   ConstraintGraph::sweep_range                 src/eval.rs:67-106
//   logup_constraint_values (D = 2 path)         src/lookup.rs:152-208
//   selectors_on_coset (p3-commit)               call src/prover.rs:775
//   shifted_quotient_slices                      src/prover.rs:631-679
//   compute_lookup_values                        src/system.rs:275-328
//   LookupValues::stage_2_traces                 src/lookup.rs:472-555
//   initial accumulator over the claims          src/prover.rs:381-387
//
// The compiled ConstraintGraph (a flat, topologically ordered node vector) is lowered on the host side of
// this library to bytecode with liveness-based slot allocation; one thread evaluates one row with its slot
// file in local memory (instructions are uniform across the warp, so the fetches broadcast). Rows of the
// committed LDEs are read where they lie: the quotient domain GENERATOR * H_{nq} is the first nq stored
// rows of every LDE in bit-reversed order, so the "current row" stream is fully coalesced.
#include "capi_common.hpp"
#include <cstdio>
#include <cstdlib>
#include "../host/blake3_host.hpp"
#include <cstring>
#include "mmcs.hpp"
#include "lowering.hpp"
#include <algorithm>
#include <cstring>

namespace msg {

}  // namespace msg

struct msgpu_program {
    msg::Ctx* ctx = nullptr;
    msg::CudaPtr<msg::Instr> d_full, d_prefix;
    u32 n_full = 0, n_prefix = 0, slots_full = 0, slots_prefix = 0;
    u32 n_zeros = 0, n_lookups = 0, n_args = 0;
    msg::CudaPtr<u32> d_zero_slots;                  // full program
    msg::CudaPtr<u32> d_mult_full, d_args_full;      // slots in the full program
    msg::CudaPtr<u32> d_mult_prefix, d_args_prefix;  // slots in the prefix program
    msg::CudaPtr<u32> d_arg_off;
    u32 pre_width = 0, main_width = 0, stage2_width = 0;
};

namespace msg {

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ gl::e2 e2_mul_k(gl::e2 x, gl::e2 y) { return gl::e2_mul(x, y); }

// a^(p-2) with 63 squarings + 10 multiplications (p - 2 = (2^32 - 2) * 2^32 + (2^32 - 1))
__device__ __forceinline__ u64 fp_inv(u64 x) {
    auto sqn = [](u64 v, int n) { for (int i = 0; i < n; i++) v = gl::mul(v, v); return v; };
    u64 t2 = gl::mul(sqn(x, 1), x);
    u64 t4 = gl::mul(sqn(t2, 2), t2);
    u64 t8 = gl::mul(sqn(t4, 4), t4);
    u64 t16 = gl::mul(sqn(t8, 8), t8);
    u64 t24 = gl::mul(sqn(t16, 8), t8);
    u64 t28 = gl::mul(sqn(t24, 4), t4);
    u64 t30 = gl::mul(sqn(t28, 2), t2);
    u64 t31 = gl::mul(sqn(t30, 1), x);
    u64 a = sqn(t31, 1);       // x^(2^32 - 2)
    u64 b = gl::mul(a, x);     // x^(2^32 - 1)
    return gl::mul(sqn(a, 32), b);
}
__device__ __forceinline__ gl::e2 e2_inverse(gl::e2 x) {
    u64 norm = gl::sub(gl::sqr(x.a), gl::mul7(gl::sqr(x.b)));
    u64 ni = fp_inv(norm);
    return gl::e2_make(gl::mul(x.a, ni), gl::mul(gl::neg(x.b), ni));
}

struct RowCtx {
    const u64* rows[3][2];  // [source][offset] -> pointer to the row
    const u64* publics;
    u64 first, last, trans;
};

// Working values of the interpreter (one per live node after liveness analysis). A per-thread array indexed by the bytecode
// lives in LOCAL memory: 256 B per thread that L1 cannot hold for a full SM, so every row's slots were written back to DRAM
// (ncu at 2^22 rows: 2.25 GB of DRAM writes for a kernel whose output is 67 MB). k_lookup_messages keeps up to 128 slots in
// shared memory instead, slot-major ([slot][thread]: conflict-free), 32 KB per 128-thread CTA at 32 slots (2.17 -> 1.68 ms);
// for k_quotient_eval the same change was a loss, its DRAM is far from saturated and the L1-resident local array is faster.
constexpr int kInterpThreads = 128;
constexpr int kSmemSlotsMax = 128;
template <int NSLOT, bool SMEM>
struct Slots;
template <int NSLOT>
struct Slots<NSLOT, false> {
    u64 v[NSLOT];
    __device__ __forceinline__ Slots() {}
    __device__ __forceinline__ u64& operator[](u32 k) { return v[k]; }
};
template <int NSLOT>
struct Slots<NSLOT, true> {
    u64* base;
    __device__ __forceinline__ Slots() {
        extern __shared__ u64 sm_slots[];
        base = sm_slots + threadIdx.x;
    }
    __device__ __forceinline__ u64& operator[](u32 k) { return base[(size_t)k * kInterpThreads]; }
};
template <int NSLOT>
constexpr size_t slots_smem_bytes() { return NSLOT <= kSmemSlotsMax ? (size_t)NSLOT * kInterpThreads * 8 : 0; }

struct NoRoots {
    __device__ __forceinline__ void operator()(u32, u64) const {}
};
template <int NSLOT, class S, class Root = NoRoots>
__device__ __forceinline__ void run_program(const Instr* __restrict__ prog, u32 n, S& slots, const RowCtx& cx, Root on_root = Root()) {
    static_assert(sizeof(Instr) == 32, "Instr must be 32 bytes");
    if (n == 0) return;
    // the next instruction is fetched while the current one executes (its fetch latency would otherwise sit on the critical
    // path of every interpreted instruction)
    uint4 nw0 = __ldg(reinterpret_cast<const uint4*>(prog));
    u64 nimm = __ldg(reinterpret_cast<const u64*>(prog) + 2);
    for (u32 pc = 0; pc < n; pc++) {
        const uint4 w0 = nw0;
        const u64 imm = nimm;
        if (pc + 1 < n) {
            nw0 = __ldg(reinterpret_cast<const uint4*>(prog + pc + 1));
            nimm = __ldg(reinterpret_cast<const u64*>(prog + pc + 1) + 2);
        }
        const u32 op = w0.x, dst = w0.y, a = w0.z, b = w0.w;
        if (op == OP_ROOT) {
            on_root((u32)imm, slots[a]);
            continue;
        }
        u64 v;
        switch (op) {
            case OP_CONST: v = imm; break;
            case OP_VAR: v = cx.rows[a & 3][a >> 2][b]; break;
            case OP_PUBLIC: v = cx.publics[a]; break;
            case OP_FIRST: v = cx.first; break;
            case OP_LAST: v = cx.last; break;
            case OP_TRANS: v = cx.trans; break;
            case OP_ADD: v = gl::add(slots[a], slots[b]); break;
            case OP_SUB: v = gl::sub(slots[a], slots[b]); break;
            case OP_MUL: v = gl::mul(slots[a], slots[b]); break;
            default: v = gl::neg(slots[a]); break;
        }
        slots[dst] = v;
    }
}

// ------------------------------------------------------------------------------------------------
// selectors on the quotient coset, in STORED (bit-reversed) order; cached per (log_n, log_q)
// ------------------------------------------------------------------------------------------------
struct SelParams {
    gl::PowTable xtab;   // 7 * w_{nq}^e
    const u64* zh;       // q entries: Z_H on the coset, indexed by i mod q
    u64 g_inv;           // w_n^{-1}
    u64* first;
    u64* last;
    u32 log_nq, log_q;
};
constexpr int kSelPerThread = 4;
__global__ void __launch_bounds__(256) k_selectors(SelParams p) {
    const u64 nq = 1ull << p.log_nq;
    u64 s0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * kSelPerThread;
    if (s0 >= nq) return;
    u64 den[2 * kSelPerThread], pref[2 * kSelPerThread], zh[kSelPerThread];
    int cnt = 0;
#pragma unroll
    for (int k = 0; k < kSelPerThread; k++) {
        u64 s = s0 + k;
        if (s >= nq) break;
        u64 i = gl::rev_bits((u32)s, p.log_nq);
        u64 x = gl::pow_lookup(p.xtab, i);
        den[2 * k] = gl::sub(x, 1);
        den[2 * k + 1] = gl::sub(x, p.g_inv);
        zh[k] = p.zh[i & ((1ull << p.log_q) - 1)];
        cnt = k + 1;
    }
    u64 acc = 1;
    for (int k = 0; k < 2 * cnt; k++) { pref[k] = acc; acc = gl::mul(acc, den[k]); }
    u64 inv = fp_inv(acc);
    for (int k = 2 * cnt; k-- > 0;) {
        u64 d = den[k];
        den[k] = gl::mul(inv, pref[k]);
        inv = gl::mul(inv, d);
    }
    for (int k = 0; k < cnt; k++) {
        p.first[s0 + k] = gl::mul(zh[k], den[2 * k]);
        p.last[s0 + k] = gl::mul(zh[k], den[2 * k + 1]);
    }
}

// ------------------------------------------------------------------------------------------------
// quotient evaluation: one thread per stored row of the quotient domain
// ------------------------------------------------------------------------------------------------
struct QuotParams {
    const Instr* prog;
    const u32* zero_slots;
    const u32 *lk_mult, *lk_argoff, *lk_args;
    const u64 *pre, *s1, *s2;
    const u64* apow;  // constraint_count x 2: weight of constraint j = alpha^{k-1-j}
    const u64 *sel_first, *sel_last, *inv_zh;
    u64* out;  // nq x 2, natural order (or n_local x 2 in stored order when out_stored)
    // Row shards (one proof over several GPUs): the cur pointers address stored rows [row0, row0 + n_local) of the quotient
    // domain, the *_n pointers the shard that holds the NEXT rows, stored rows [next_row0, ...). Unsharded: row0 = next_row0 = 0,
    // n_local = nq and the next pointers equal the cur ones.
    const u64 *pre_n, *s1_n, *s2_n;
    u32 wn[3], cn[3];  // the next buffers' row strides and first columns (a shard may fetch only the columns read at the next row)
    u64 row0, n_local, next_row0;
    u32 out_stored;
    gl::PowTable xtab;
    u64 publics[8];
    u64 delta[2];
    u64 g_inv;
    u32 n_instr, n_zeros, n_lookups;
    u32 wpre, w1, w2;
    u32 log_nq, log_q;
};

template <int NSLOT>
__global__ void __launch_bounds__(128) k_quotient_eval(QuotParams p) {
    const u64 nq = 1ull << p.log_nq;
    const u64 sl = (u64)blockIdx.x * blockDim.x + threadIdx.x;  // local row
    if (sl >= p.n_local) return;
    const u64 s = p.row0 + sl;
    const u64 i = gl::rev_bits((u32)s, p.log_nq);
    const u64 inext = (i + (1ull << p.log_q)) & (nq - 1);
    const u64 sn = gl::rev_bits((u32)inext, p.log_nq) - p.next_row0;  // inside the shard the next pointers address
    RowCtx cx;
    cx.rows[0][0] = p.pre + sl * p.wpre;
    cx.rows[0][1] = p.pre_n + sn * p.wn[0] - p.cn[0];
    cx.rows[1][0] = p.s1 + sl * p.w1;
    cx.rows[1][1] = p.s1_n + sn * p.wn[1] - p.cn[1];
    cx.rows[2][0] = p.s2 + sl * p.w2;
    cx.rows[2][1] = p.s2_n + sn * p.wn[2] - p.cn[2];
    cx.publics = p.publics;
    cx.first = p.sel_first[s];
    cx.last = p.sel_last[s];
    cx.trans = gl::sub(gl::pow_lookup(p.xtab, i), p.g_inv);
    Slots<NSLOT, false> slots;  // measured: shared-memory slots make THIS kernel slower (1.83 -> 2.58 ms at 2^22 rows), local ones stay
    // alpha-fold with lazy 160-bit accumulation: one reduction per coordinate at the end. Constraint j of the DAG is folded by
    // the OP_ROOT instruction that follows its node (weight apow[j]); the logUp constraints continue at index n_zeros.
    gl::Acc160 fa0 = gl::acc_zero(), fa1 = gl::acc_zero();
    run_program<NSLOT>(p.prog, p.n_instr, slots, cx, [&](u32 j, u64 v) {
        gl::acc_mac(fa0, v, __ldg(p.apow + 2 * j));
        gl::acc_mac(fa1, v, __ldg(p.apow + 2 * j + 1));
    });
    u32 ci = p.n_zeros;
    // logUp constraint values (src/lookup.rs:167-208)
    const u64* s2c = cx.rows[2][0];
    const u64* s2n = cx.rows[2][1];
    const gl::e2 beta = gl::e2_make(p.publics[0], p.publics[1]), gamma = gl::e2_make(p.publics[2], p.publics[3]);
    const gl::e2 inj = gl::e2_make(gl::mul(cx.last, p.delta[0]), gl::mul(cx.last, p.delta[1]));
    auto fold = [&](u64 v) {
        gl::acc_mac(fa0, v, __ldg(p.apow + 2 * ci));
        gl::acc_mac(fa1, v, __ldg(p.apow + 2 * ci + 1));
        ci++;
    };
    if (p.n_lookups == 0) {
        fold(gl::add(gl::sub(s2n[0], s2c[0]), inj.a));
        fold(gl::add(gl::sub(s2n[1], s2c[1]), inj.b));
    } else {
        for (u32 j = 0; j < p.n_lookups; j++) {
            gl::e2 source = gl::e2_make(s2c[2 * j], s2c[2 * j + 1]);
            gl::e2 target = j + 1 < p.n_lookups ? gl::e2_make(s2c[2 * j + 2], s2c[2 * j + 3])
                                                : gl::e2_make(gl::add(s2n[0], inj.a), gl::add(s2n[1], inj.b));
            gl::e2 f = gl::e2_make(0, 0);
            for (u32 k = p.lk_argoff[j + 1]; k-- > p.lk_argoff[j];) {
                f = gl::e2_mul(f, gamma);
                f.a = gl::add(f.a, slots[p.lk_args[k]]);
            }
            gl::e2 c = gl::e2_mul(gl::e2_add(f, beta), gl::e2_sub(target, source));
            fold(gl::sub(c.a, slots[p.lk_mult[j]]));
            fold(c.b);
        }
    }
    const u64 iv = p.inv_zh[i & ((1ull << p.log_q) - 1)];
    const u64 o = p.out_stored ? sl : i;
    p.out[2 * o] = gl::mul(gl::acc_reduce(fa0), iv);
    p.out[2 * o + 1] = gl::mul(gl::acc_reduce(fa1), iv);
}

// out[r][k*d + c] = S[rev((N - (k*n + r)) mod N)][c] * weights[k]     (src/prover.rs:659-677)
__global__ void k_quotient_slices(const u64* S, u64* out, u32 log_big, u32 log_n, u32 d, const u64* weights) {
    const u64 big = 1ull << log_big, n = 1ull << log_n, q = big >> log_n;
    u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= big) return;
    u64 r = t / q, k = t % q;
    u64 j = k * n + r;
    u64 src = gl::rev_bits((u32)((big - j) & (big - 1)), log_big);
    u64 w = weights[k];
    for (u32 c = 0; c < d; c++) out[r * (q * d) + k * d + c] = gl::mul(S[src * d + c], w);
}

// ------------------------------------------------------------------------------------------------
// stage-2 trace construction
// ------------------------------------------------------------------------------------------------
struct MsgParams {
    const Instr* prog;
    const u32 *lk_mult, *lk_argoff, *lk_args;
    const u64 *pre, *main;
    u64* msgs;   // rows * L x 2
    u64* mults;  // rows * L
    u64 rows;
    u64 beta[2], gamma[2];
    u32 n_instr, n_lookups, wpre, wmain;
};
template <int NSLOT>
__global__ void __launch_bounds__(128) k_lookup_messages(MsgParams p) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= p.rows) return;
    const u64 rn = r + 1 == p.rows ? 0 : r + 1;
    RowCtx cx;
    cx.rows[0][0] = p.pre + r * p.wpre;
    cx.rows[0][1] = p.pre + rn * p.wpre;
    cx.rows[1][0] = p.main + r * p.wmain;
    cx.rows[1][1] = p.main + rn * p.wmain;
    cx.rows[2][0] = cx.rows[2][1] = nullptr;  // lookup expressions cannot read stage 2 or publics (refused by program_create)
    cx.publics = nullptr;
    cx.first = r == 0;
    cx.last = r + 1 == p.rows;
    cx.trans = r + 1 != p.rows;
    Slots<NSLOT, (NSLOT <= kSmemSlotsMax)> slots;
    run_program<NSLOT>(p.prog, p.n_instr, slots, cx);
    const gl::e2 beta = gl::e2_make(p.beta[0], p.beta[1]), gamma = gl::e2_make(p.gamma[0], p.gamma[1]);
    for (u32 j = 0; j < p.n_lookups; j++) {
        gl::e2 f = gl::e2_make(0, 0);
        for (u32 k = p.lk_argoff[j + 1]; k-- > p.lk_argoff[j];) {
            f = gl::e2_mul(f, gamma);
            f.a = gl::add(f.a, slots[p.lk_args[k]]);
        }
        f = gl::e2_add(f, beta);
        u64 idx = r * p.n_lookups + j;
        p.msgs[2 * idx] = f.a;
        p.msgs[2 * idx + 1] = f.b;
        p.mults[idx] = slots[p.lk_mult[j]];
    }
}

constexpr int kScanPerThread = 8;
constexpr int kScanThreads = 256;
constexpr int kScanPerBlock = kScanPerThread * kScanThreads;

// block reduction of extension values; result valid in thread 0
__device__ __forceinline__ gl::e2 block_sum(gl::e2 v, gl::e2* sm) {
    for (int off = 16; off > 0; off >>= 1) {
        v.a = gl::add(v.a, __shfl_down_sync(0xffffffffu, v.a, off));
        v.b = gl::add(v.b, __shfl_down_sync(0xffffffffu, v.b, off));
    }
    int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) sm[wid] = v;
    __syncthreads();
    gl::e2 r = gl::e2_make(0, 0);
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) r = gl::e2_add(r, sm[w]);
    return r;
}

// msgs[i] <- mults[i] / msgs[i] (Montgomery batches of 8 per thread); block_sums[b] = sum of the block's terms. A zero message
// (the batch product is zero only then: 7 is a non-residue, so only 0 has norm 0) sets *zero_msg instead of a silent 0 inverse.
__global__ void __launch_bounds__(kScanThreads) k_terms_and_block_sums(u64* msgs, const u64* mults, u64 total, u64* block_sums,
                                                                       u64* zero_msg) {
    __shared__ gl::e2 sm[kScanThreads / 32];
    u64 i0 = ((u64)blockIdx.x * kScanThreads + threadIdx.x) * kScanPerThread;
    // prefix products in registers (fully unrolled, constant indices: a dynamically indexed array would live in local memory,
    // 256 B per thread that ends up in DRAM); the messages themselves are read a second time on the way back (L1 / L2 hits)
    gl::e2 pref[kScanPerThread];
    const int cnt = (int)min((u64)kScanPerThread, total > i0 ? total - i0 : 0);
    gl::e2 acc = gl::e2_make(1, 0);
#pragma unroll
    for (int k = 0; k < kScanPerThread; k++) {
        pref[k] = acc;
        if (k < cnt) acc = gl::e2_mul(acc, gl::e2_make(msgs[2 * (i0 + k)], msgs[2 * (i0 + k) + 1]));
    }
    if (cnt && acc.a == 0 && acc.b == 0) *zero_msg = 1;
    gl::e2 inv = cnt ? e2_inverse(acc) : acc;
    gl::e2 sum = gl::e2_make(0, 0);
#pragma unroll
    for (int k = kScanPerThread - 1; k >= 0; k--) {
        if (k < cnt) {
            gl::e2 x = gl::e2_make(msgs[2 * (i0 + k)], msgs[2 * (i0 + k) + 1]);
            gl::e2 xi = gl::e2_mul(inv, pref[k]);
            inv = gl::e2_mul(inv, x);
            gl::e2 term = gl::e2_mul_base(xi, mults[i0 + k]);
            msgs[2 * (i0 + k)] = term.a;
            msgs[2 * (i0 + k) + 1] = term.b;
            sum = gl::e2_add(sum, term);
        }
    }
    gl::e2 bs = block_sum(sum, sm);
    if (threadIdx.x == 0) { block_sums[2 * blockIdx.x] = bs.a; block_sums[2 * blockIdx.x + 1] = bs.b; }
}

// in-place exclusive scan of the block sums (single block); total written after the last element
__global__ void __launch_bounds__(1024) k_scan_block_sums(u64* block_sums, u64 nblocks) {
    __shared__ gl::e2 sm[1024];
    // each thread owns a contiguous chunk
    u64 per = (nblocks + blockDim.x - 1) / blockDim.x;
    u64 lo = (u64)threadIdx.x * per, hi = min(nblocks, lo + per);
    gl::e2 s = gl::e2_make(0, 0);
    for (u64 i = lo; i < hi; i++) s = gl::e2_add(s, gl::e2_make(block_sums[2 * i], block_sums[2 * i + 1]));
    sm[threadIdx.x] = s;
    __syncthreads();
    // Hillis-Steele inclusive scan over the 1024 chunk sums
    for (int off = 1; off < (int)blockDim.x; off <<= 1) {
        gl::e2 t = sm[threadIdx.x];
        if ((int)threadIdx.x >= off) t = gl::e2_add(t, sm[threadIdx.x - off]);
        __syncthreads();
        sm[threadIdx.x] = t;
        __syncthreads();
    }
    gl::e2 run = threadIdx.x ? sm[threadIdx.x - 1] : gl::e2_make(0, 0);
    for (u64 i = lo; i < hi; i++) {
        gl::e2 v = gl::e2_make(block_sums[2 * i], block_sums[2 * i + 1]);
        block_sums[2 * i] = run.a;
        block_sums[2 * i + 1] = run.b;
        run = gl::e2_add(run, v);
    }
    if (threadIdx.x == blockDim.x - 1) {
        gl::e2 tot = sm[blockDim.x - 1];
        block_sums[2 * nblocks] = tot.a;
        block_sums[2 * nblocks + 1] = tot.b;
    }
}

// out[i] = block_offset + exclusive prefix of terms within the block
__global__ void __launch_bounds__(kScanThreads) k_scan_write(const u64* terms, u64 total, const u64* block_offsets, u64* out) {
    __shared__ gl::e2 sm[kScanThreads];
    u64 i0 = ((u64)blockIdx.x * kScanThreads + threadIdx.x) * kScanPerThread;
    gl::e2 v[kScanPerThread];
    gl::e2 s = gl::e2_make(0, 0);
    for (int k = 0; k < kScanPerThread; k++) {
        v[k] = i0 + k < total ? gl::e2_make(terms[2 * (i0 + k)], terms[2 * (i0 + k) + 1]) : gl::e2_make(0, 0);
        s = gl::e2_add(s, v[k]);
    }
    sm[threadIdx.x] = s;
    __syncthreads();
    for (int off = 1; off < kScanThreads; off <<= 1) {
        gl::e2 t = sm[threadIdx.x];
        if ((int)threadIdx.x >= off) t = gl::e2_add(t, sm[threadIdx.x - off]);
        __syncthreads();
        sm[threadIdx.x] = t;
        __syncthreads();
    }
    gl::e2 run = gl::e2_make(block_offsets[2 * blockIdx.x], block_offsets[2 * blockIdx.x + 1]);
    if (threadIdx.x) run = gl::e2_add(run, sm[threadIdx.x - 1]);
    for (int k = 0; k < kScanPerThread; k++) {
        if (i0 + k >= total) break;
        out[2 * (i0 + k)] = run.a;
        out[2 * (i0 + k) + 1] = run.b;
        run = gl::e2_add(run, v[k]);
    }
}

// partial[b] = sum over the block's claims of 1 / (beta + fingerprint(gamma, claim)); a zero message sets *zero_msg
__global__ void __launch_bounds__(kScanThreads) k_claims(const u64* claims, u64 n_claims, u32 len, gl::e2 beta, gl::e2 gamma,
                                                         u64* partial, u64* zero_msg) {
    __shared__ gl::e2 sm[kScanThreads / 32];
    u64 i0 = ((u64)blockIdx.x * kScanThreads + threadIdx.x) * kScanPerThread;
    // fully unrolled, constant indices: the batch of 8 stays in registers
    const int cnt = (int)min((u64)kScanPerThread, n_claims > i0 ? n_claims - i0 : 0);
    gl::e2 v[kScanPerThread], pref[kScanPerThread];
    gl::e2 acc = gl::e2_make(1, 0);
#pragma unroll
    for (int k = 0; k < kScanPerThread; k++) {
        pref[k] = acc;
        v[k] = acc;
        if (k < cnt) {
            const u64* c = claims + (i0 + k) * len;
            gl::e2 f = gl::e2_make(0, 0);
            for (u32 a = len; a-- > 0;) {
                f = gl::e2_mul(f, gamma);
                f.a = gl::add(f.a, c[a]);
            }
            v[k] = gl::e2_add(f, beta);
            acc = gl::e2_mul(acc, v[k]);
        }
    }
    if (cnt && acc.a == 0 && acc.b == 0) *zero_msg = 1;
    gl::e2 inv = cnt ? e2_inverse(acc) : acc;
    gl::e2 sum = gl::e2_make(0, 0);
#pragma unroll
    for (int k = kScanPerThread - 1; k >= 0; k--) {
        if (k < cnt) {
            sum = gl::e2_add(sum, gl::e2_mul(inv, pref[k]));
            inv = gl::e2_mul(inv, v[k]);
        }
    }
    gl::e2 bs = block_sum(sum, sm);
    if (threadIdx.x == 0) { partial[2 * blockIdx.x] = bs.a; partial[2 * blockIdx.x + 1] = bs.b; }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
template <class T>
static CudaPtr<T> upload_vec(Ctx& c, const std::vector<T>& v) {
    CudaPtr<T> d = cuda_malloc<T>(std::max<size_t>(v.size(), 1));
    if (!v.empty()) MSG_CUDA(cudaMemcpyAsync(d.get(), v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, c.stream));
    return d;
}

static std::unique_ptr<msgpu_program> program_create(Ctx& c, const msgpu_graph_desc& g) {
    MSG_REQUIRE(g.lookup_prefix_len <= g.n_nodes, "program: lookup prefix longer than the node vector");
    MSG_REQUIRE(g.stage2_width == 2 * std::max<u32>(g.n_lookups, 1), "program: stage-2 width must be 2 * max(lookups, 1)");
    // k_lookup_messages has no stage-2 rows and no publics: lookup values are computed before either exists
    for (u32 i = 0; i < g.lookup_prefix_len; i++) {
        MSG_REQUIRE(g.op[i] != OP_PUBLIC, "program: lookup expression reads a public value");
        MSG_REQUIRE(g.op[i] != OP_VAR || (g.a[i] & 3) != 2, "program: lookup expression reads a stage-2 column");
    }
    std::vector<u32> pin_lk, pin_all;
    u32 n_args = g.n_lookups ? g.lookup_arg_off[g.n_lookups] : 0;
    for (u32 j = 0; j < g.n_lookups; j++) pin_lk.push_back(g.lookup_mult[j]);
    for (u32 k = 0; k < n_args; k++) pin_lk.push_back(g.lookup_args[k]);
    pin_all = pin_lk;
    std::vector<u32> roots(g.zeros, g.zeros + g.n_zeros);
    for (u32 p : pin_lk) MSG_REQUIRE(p < g.lookup_prefix_len, "program: lookup node outside the prefix");
    Lowered full, prefix;
    try {
        full = lower(g, g.n_nodes, pin_all, roots);
        prefix = lower(g, g.lookup_prefix_len, pin_lk);
    } catch (const LowerError& e) {
        throw Error(MSGPU_ERR_INVALID, e.what());
    }
    MSG_REQUIRE(full.n_slots <= 4096 && prefix.n_slots <= 4096, "program: circuit needs more than 4096 live values");
    if (getenv("MSGPU_TIMELINE"))
        fprintf(stderr, "[program] %u nodes, %u roots, %u lookups: full program %zu instructions / %u slots, lookup prefix %zu / %u\n", g.n_nodes,
                g.n_zeros, g.n_lookups, full.code.size(), full.n_slots, prefix.code.size(), prefix.n_slots);
    auto prog = std::make_unique<msgpu_program>();
    prog->ctx = &c;
    prog->n_full = (u32)full.code.size();
    prog->n_prefix = (u32)prefix.code.size();
    prog->slots_full = full.n_slots;
    prog->slots_prefix = prefix.n_slots;
    prog->n_zeros = g.n_zeros;
    prog->n_lookups = g.n_lookups;
    prog->n_args = n_args;
    prog->pre_width = g.pre_width;
    prog->main_width = g.main_width;
    prog->stage2_width = g.stage2_width;
    prog->d_full = upload_vec(c, full.code);
    prog->d_prefix = upload_vec(c, prefix.code);
    std::vector<u32> zs, mf, af, mp, ap, off;
    zs.assign(std::max<u32>(g.n_zeros, 1), 0);  // (the roots are folded by OP_ROOT instructions; kept for the layout)
    for (u32 j = 0; j < g.n_lookups; j++) { mf.push_back(full.slot_of[g.lookup_mult[j]]); mp.push_back(prefix.slot_of[g.lookup_mult[j]]); }
    for (u32 k = 0; k < n_args; k++) { af.push_back(full.slot_of[g.lookup_args[k]]); ap.push_back(prefix.slot_of[g.lookup_args[k]]); }
    for (u32 j = 0; j <= g.n_lookups; j++) off.push_back(g.n_lookups ? g.lookup_arg_off[j] : 0);
    prog->d_zero_slots = upload_vec(c, zs);
    prog->d_mult_full = upload_vec(c, mf);
    prog->d_args_full = upload_vec(c, af);
    prog->d_mult_prefix = upload_vec(c, mp);
    prog->d_args_prefix = upload_vec(c, ap);
    prog->d_arg_off = upload_vec(c, off);
    c.sync();
    return prog;
}

using SelCache = Ctx::SelCache;

static gl::PowTable coset_x_table(Ctx& c, u32 log_nq) {
    return c.pow_table(msh::two_adic_generator(log_nq).v, msh::GL_GENERATOR, log_nq).view();
}

static const SelCache& selectors(Ctx& c, u32 log_n, u32 log_q) {
    auto& cache = c.sel_cache;
    auto key = std::make_pair(log_n, log_q);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    u32 log_nq = log_n + log_q;
    u64 nq = 1ull << log_nq, q = 1ull << log_q;
    std::vector<u64> zh(q), izh(q);
    msh::Fp s_pow_n = msh::Fp(msh::GL_GENERATOR).exp_power_of_2(log_n), wq = msh::two_adic_generator(log_q), acc = msh::Fp::one();
    for (u64 i = 0; i < q; i++) {
        msh::Fp z = s_pow_n * acc - msh::Fp::one();
        zh[i] = z.v;
        izh[i] = z.inverse().v;
        acc *= wq;
    }
    SelCache sc{cuda_malloc<u64>(nq), cuda_malloc<u64>(nq), cuda_malloc<u64>(q), cuda_malloc<u64>(q)};
    MSG_CUDA(cudaMemcpyAsync(sc.zh.get(), zh.data(), q * 8, cudaMemcpyHostToDevice, c.stream));
    MSG_CUDA(cudaMemcpyAsync(sc.inv_zh.get(), izh.data(), q * 8, cudaMemcpyHostToDevice, c.stream));
    SelParams sp{};
    sp.xtab = coset_x_table(c, log_nq);
    sp.zh = sc.zh.get();
    sp.g_inv = msh::two_adic_generator(log_n).inverse().v;
    sp.first = sc.first.get();
    sp.last = sc.last.get();
    sp.log_nq = log_nq;
    sp.log_q = log_q;
    u64 threads = (nq + kSelPerThread - 1) / kSelPerThread;
    {
        StageScope ss(c, "quotient");
        launch(c, "k_selectors", k_selectors, (unsigned)((threads + 255) / 256), 256, 0, sp);
    }
    c.sync();  // zh / izh host vectors die here
    return cache[key] = std::move(sc);
}

template <class K>
static void launch_by_slots(u32 n_slots, K&& launch) {
    if (n_slots <= 32) launch(std::integral_constant<int, 32>());
    else if (n_slots <= 64) launch(std::integral_constant<int, 64>());
    else if (n_slots <= 128) launch(std::integral_constant<int, 128>());
    else if (n_slots <= 256) launch(std::integral_constant<int, 256>());
    else if (n_slots <= 1024) launch(std::integral_constant<int, 1024>());
    else launch(std::integral_constant<int, 4096>());
}

static void quotient_slices(Ctx& c, const u64* S, u64* out, u32 log_big, u32 log_n, u32 d) {
    u64 big = 1ull << log_big, n = 1ull << log_n, q = big >> log_n;
    std::vector<u64> w(q);
    msh::Fp ninv = msh::Fp((msh::u64)big).inverse();
    msh::Fp step = msh::Fp(msh::GL_GENERATOR).pow((msh::u64)n).inverse(), acc = msh::Fp::one();
    for (u64 k = 0; k < q; k++) { w[k] = (acc * ninv).v; acc *= step; }
    DevBuf dw(c, q * 8);
    MSG_CUDA(cudaMemcpyAsync(dw.p, w.data(), q * 8, cudaMemcpyHostToDevice, c.stream));
    launch(c, "k_quotient_slices", k_quotient_slices, (unsigned)((big + 255) / 256), 256, 0, S, out, log_big, log_n, d, (const u64*)dw.u());
    c.sync();  // `w` dies here (pageable source of an async copy)
}

static void view_of(const msgpu_pdata* pd, u64 idx, u64 nq, u32 width, const u64** ptr) {
    MSG_REQUIRE(pd && idx < pd->mats.size(), "quotient: matrix index out of range");
    auto& m = pd->mats[idx];
    MSG_REQUIRE(m.width == width, "quotient: committed width does not match the program");
    MSG_REQUIRE(m.height >= nq, "quotient: quotient domain larger than the committed LDE (quotient degree > blowup)");
    *ptr = m.ptr;
}

}  // namespace msg

using namespace msg;

struct msgpu_claims {
    Ctx* ctx;
    DevBuf d;
    u64 n, len;
    Event ready;  // prefetched claims: the copy on the context's copy stream has finished
};

namespace msg {
// msg[prefix_len + 8*j ..] = le64(word j), word j of claim i = j / (len+1): position 0 is the length, then the values
__global__ void __launch_bounds__(256) k_encode_claims(const u64* claims, u64 n_words, u32 len, uint8_t* msg) {
    u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_words) return;
    u64 claim = j / (len + 1);
    u32 k = (u32)(j % (len + 1));
    u64 v = k == 0 ? (u64)len : claims[claim * len + (k - 1)];
    uint8_t* o = msg + 8 * j;
#pragma unroll
    for (int b = 0; b < 8; b++) o[b] = (uint8_t)(v >> (8 * b));
}
}  // namespace msg

static void claims_sum(Ctx& c, const u64* d_claims, u64 n_claims, u64 claim_len, const uint64_t* beta2, const uint64_t* gamma2,
                       uint64_t* out2) {
    StageScope ss(c, "stage2");
    out2[0] = out2[1] = 0;
    if (n_claims == 0) return;
    u64 nblocks = (n_claims + kScanPerBlock - 1) / kScanPerBlock;
    DevBuf part(c, nblocks * 16 + 8);  // the block partials, then the zero-message flag
    MSG_CUDA(cudaMemsetAsync(part.u() + 2 * nblocks, 0, 8, c.stream));
    launch(c, "k_claims", k_claims, (unsigned)nblocks, kScanThreads, 0, d_claims, n_claims, (u32)claim_len, gl::e2{beta2[0], beta2[1]},
           gl::e2{gamma2[0], gamma2[1]}, part.u(), part.u() + 2 * nblocks);
    std::vector<u64> hp(nblocks * 2 + 1);
    MSG_CUDA(cudaMemcpyAsync(hp.data(), part.p, nblocks * 16 + 8, cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    MSG_REQUIRE(hp[2 * nblocks] == 0, "claims: a logUp message beta + fingerprint(gamma, claim) is zero");
    msh::Fp2 acc;
    for (u64 b = 0; b < nblocks; b++) acc += msh::Fp2(msh::Fp(hp[2 * b]), msh::Fp(hp[2 * b + 1]));
    out2[0] = acc.c[0].v;
    out2[1] = acc.c[1].v;
}

extern "C" {

int msgpu_program_create(msgpu_ctx* h, const msgpu_graph_desc* desc, msgpu_program** out) {
    return guard([&] {
        MSG_REQUIRE(desc && out, "program_create: null argument");
        *out = program_create(h->c, *desc).release();
    });
}
void msgpu_program_free(msgpu_program* prog) {
    if (!prog) return;
    cudaStreamSynchronize(prog->ctx->stream);
    delete prog;
}

int msgpu_stage2_trace(msgpu_ctx* h, const msgpu_program* prog, const uint64_t* pre_dev, const uint64_t* main_dev,
                       uint64_t rows, const uint64_t* beta2, const uint64_t* gamma2, uint64_t* stage2_out_dev,
                       uint64_t* local_sum2) {
    return guard([&] {
        Ctx& c = h->c;
        StageScope ss(c, "stage2");
        MSG_REQUIRE(prog && stage2_out_dev && local_sum2, "stage2_trace: null argument");
        MSG_REQUIRE(main_dev || prog->n_lookups == 0, "stage2_trace: the main trace is needed to evaluate the lookups");
        MSG_REQUIRE(prog->pre_width == 0 || pre_dev, "stage2_trace: circuit has a preprocessed trace but none was given");
        local_sum2[0] = local_sum2[1] = 0;
        if (rows == 0) return;
        u32 L = prog->n_lookups;
        if (L == 0) {  // pass-through accumulator column, zero by convention (src/lookup.rs:520-524)
            MSG_CUDA(cudaMemsetAsync(stage2_out_dev, 0, rows * 2 * 8, c.stream));
            return;
        }
        u64 total = rows * L;
        u64 nblocks = (total + kScanPerBlock - 1) / kScanPerBlock;
        // bsums: the block sums, the total, then the zero-message flag
        DevBuf msgs(c, total * 16), mults(c, total * 8), bsums(c, (nblocks + 1) * 16 + 8);
        u64* zero_msg = bsums.u() + 2 * (nblocks + 1);
        MSG_CUDA(cudaMemsetAsync(zero_msg, 0, 8, c.stream));
        MsgParams mp{};
        mp.prog = prog->d_prefix.get();
        mp.n_instr = prog->n_prefix;
        mp.lk_mult = prog->d_mult_prefix.get();
        mp.lk_argoff = prog->d_arg_off.get();
        mp.lk_args = prog->d_args_prefix.get();
        mp.pre = (const u64*)pre_dev;
        mp.main = (const u64*)main_dev;
        mp.msgs = msgs.u();
        mp.mults = mults.u();
        mp.rows = rows;
        mp.beta[0] = beta2[0]; mp.beta[1] = beta2[1];
        mp.gamma[0] = gamma2[0]; mp.gamma[1] = gamma2[1];
        mp.n_lookups = L;
        mp.wpre = prog->pre_width;
        mp.wmain = prog->main_width;
        launch_by_slots(prog->slots_prefix, [&](auto ns) {
            constexpr int NS = decltype(ns)::value;
            constexpr size_t smem = slots_smem_bytes<NS>();
            if (smem > 48 * 1024) ensure_max_smem(k_lookup_messages<NS>, (int)smem);
            launch(c, "k_lookup_messages", k_lookup_messages<NS>, (unsigned)((rows + 127) / 128), kInterpThreads, smem, mp);
        });
        launch(c, "k_terms_and_block_sums", k_terms_and_block_sums, (unsigned)nblocks, kScanThreads, 0, msgs.u(), mults.u(), total, bsums.u(),
               zero_msg);
        launch(c, "k_scan_block_sums", k_scan_block_sums, 1, 1024, 0, bsums.u(), nblocks);
        launch(c, "k_scan_write", k_scan_write, (unsigned)nblocks, kScanThreads, 0, msgs.u(), total, bsums.u(), (u64*)stage2_out_dev);
        u64 tail[3];  // total, zero-message flag
        MSG_CUDA(cudaMemcpyAsync(tail, bsums.u() + 2 * nblocks, 24, cudaMemcpyDeviceToHost, c.stream));
        c.sync();
        MSG_REQUIRE(tail[2] == 0, "stage2_trace: a logUp message beta + fingerprint(gamma, args) is zero");
        local_sum2[0] = tail[0];
        local_sum2[1] = tail[1];
    });
}

int msgpu_claims_accumulator(msgpu_ctx* h, const uint64_t* claims, uint64_t n_claims, uint64_t claim_len,
                             const uint64_t* beta2, const uint64_t* gamma2, uint64_t* out2) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(claim_len < (1ull << 31), "claims: claim too long");
        DevBuf d(c, n_claims * std::max<u64>(claim_len, 1) * 8);
        if (claim_len && n_claims) MSG_CUDA(cudaMemcpyAsync(d.p, claims, n_claims * claim_len * 8, cudaMemcpyHostToDevice, c.stream));
        claims_sum(c, d.u(), n_claims, claim_len, beta2, gamma2, out2);
    });
}

// BLAKE3(prefix || encoded claims) of device-resident claims + the canonical check (shared by upload and digest)
static void claims_digest(Ctx& c, const u64* d_claims, u64 n_claims, u64 claim_len, const uint8_t* prefix, u64 prefix_len, uint8_t* digest32);

int msgpu_claims_upload(msgpu_ctx* h, const uint64_t* claims, uint64_t n_claims, uint64_t claim_len, const uint8_t* prefix,
                        uint64_t prefix_len, msgpu_claims** out, uint8_t* digest32) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(out && digest32 && claims && n_claims > 0 && claim_len > 0, "claims_upload: null or empty argument");
        MSG_REQUIRE(claim_len < (1ull << 31) && n_claims <= (~0ull) / 16 / (claim_len + 1), "claims_upload: too large");
        u64 n_vals = n_claims * claim_len;
        DevBuf d(c, n_vals * 8);
        MSG_CUDA(cudaMemcpyAsync(d.p, claims, n_vals * 8, cudaMemcpyHostToDevice, c.stream));
        claims_digest(c, d.u(), n_claims, claim_len, prefix, prefix_len, digest32);
        *out = new msgpu_claims{&c, std::move(d), n_claims, claim_len, Event()};
    });
}

int msgpu_claims_prefetch(msgpu_ctx* h, const uint64_t* claims, uint64_t n_claims, uint64_t claim_len, msgpu_claims** out) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(out && claims && n_claims > 0 && claim_len > 0, "claims_prefetch: null or empty argument");
        MSG_REQUIRE(claim_len < (1ull << 31) && n_claims <= (~0ull) / 16 / (claim_len + 1), "claims_prefetch: too large");
        if (!c.copy_stream) MSG_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
        u64 n_vals = n_claims * claim_len;
        DevBuf d(c, n_vals * 8);
        // the copy starts behind everything already enqueued on the main stream (the block may have just been freed by it,
        // and the trace upload should have the link to itself) and runs under whatever the main stream does next
        auto cl = std::unique_ptr<msgpu_claims>(new msgpu_claims{&c, std::move(d), n_claims, claim_len, Event()});
        cudaEvent_t e0;
        MSG_CUDA(cudaEventCreateWithFlags(&e0, cudaEventDisableTiming));
        MSG_CUDA(cudaEventRecord(e0, c.stream));
        MSG_CUDA(cudaStreamWaitEvent(c.copy_stream, e0, 0));
        cudaEventDestroy(e0);
        MSG_CUDA(cudaMemcpyAsync(cl->d.p, claims, n_vals * 8, cudaMemcpyHostToDevice, c.copy_stream));
        cl->ready.record(c.copy_stream);
        *out = cl.release();
    });
}

int msgpu_claims_digest(msgpu_claims* cl, const uint8_t* prefix, uint64_t prefix_len, uint8_t* digest32) {
    return guard([&] {
        MSG_REQUIRE(cl && digest32, "claims_digest: null argument");
        Ctx& c = *cl->ctx;
        if (cl->ready.e) MSG_CUDA(cudaStreamWaitEvent(c.stream, cl->ready.e, 0));
        claims_digest(c, cl->d.u(), cl->n, cl->len, prefix, prefix_len, digest32);
    });
}

static void claims_digest(Ctx& c, const u64* d_claims, u64 n_claims, u64 claim_len, const uint8_t* prefix, u64 prefix_len, uint8_t* digest32) {
    {
        StageScope ss(c, "transcript");
        u64 n_vals = n_claims * claim_len, n_words = n_claims * (claim_len + 1), msg_len = prefix_len + 8 * n_words;
        DevBuf msg(c, msg_len + 64), flag(c, 4);
        struct { const u64* p; const u64* u() const { return p; } } d{d_claims};
        MSG_CUDA(cudaMemsetAsync(flag.p, 0, 4, c.stream));
        check_canonical(c, d.u(), n_vals, (u32*)flag.p);
        if (prefix_len) MSG_CUDA(cudaMemcpyAsync(msg.p, prefix, prefix_len, cudaMemcpyHostToDevice, c.stream));
        launch(c, "k_encode_claims", k_encode_claims, (unsigned)((n_words + 255) / 256), 256, 0, d.u(), n_words, (u32)claim_len,
               msg.bytes() + prefix_len);
        u32 bad = 0;
        if (msg_len > 1024) {
            uint8_t* out_dev = (uint8_t*)msg.p + ((msg_len + 15) / 16) * 16;
            b3_hash_long(c, (const uint8_t*)msg.p, msg_len, out_dev);
            MSG_CUDA(cudaMemcpyAsync(digest32, out_dev, 32, cudaMemcpyDeviceToHost, c.stream));
            MSG_CUDA(cudaMemcpyAsync(&bad, flag.p, 4, cudaMemcpyDeviceToHost, c.stream));
            c.sync();
        } else {
            std::vector<uint8_t> hm(msg_len);
            MSG_CUDA(cudaMemcpyAsync(hm.data(), msg.p, msg_len, cudaMemcpyDeviceToHost, c.stream));
            MSG_CUDA(cudaMemcpyAsync(&bad, flag.p, 4, cudaMemcpyDeviceToHost, c.stream));
            c.sync();
            msh::Digest dg = msh::blake3_hash(hm.data(), hm.size());
            memcpy(digest32, dg.data(), 32);
        }
        MSG_REQUIRE(bad == 0, "claims_upload: claim value is not a canonical field element (>= p)");
    }
}
int msgpu_claims_accumulate(msgpu_claims* cl, const uint64_t* beta2, const uint64_t* gamma2, uint64_t* out2) {
    return guard([&] {
        MSG_REQUIRE(cl && beta2 && gamma2 && out2, "claims_accumulate: null argument");
        if (cl->ready.e) MSG_CUDA(cudaStreamWaitEvent(cl->ctx->stream, cl->ready.e, 0));
        claims_sum(*cl->ctx, cl->d.u(), cl->n, cl->len, beta2, gamma2, out2);
    });
}
void msgpu_claims_free(msgpu_claims* cl) { delete cl; }

}  // extern "C"

namespace msg {
// k_quotient_eval over stored rows [row0, row0 + n_local) of the quotient domain. cur[3] / nxt[3]: pre, stage 1, stage 2 row
// pointers of the local rows / of the shard holding the next rows (first stored row next_row0).
static void quotient_eval(Ctx& c, const msgpu_program* prog, const u64* const cur[3], const u64* const nxt[3], u64 row0, u64 n_local,
                          u64 next_row0, u32 log_n, u32 log_q, const uint64_t* publics8, const uint64_t* alpha2, u64* out, bool out_stored,
                          const u32* next_widths3 = nullptr, const u32* next_col0_3 = nullptr) {
    const u32 log_nq = log_n + log_q;
    const u64 n = 1ull << log_n;
    for (int i = 0; i < 8; i++) MSG_REQUIRE(publics8[i] < GLD_P, "quotient: public value is not canonical");
    QuotParams qp{};
    qp.pre = cur[0]; qp.s1 = cur[1]; qp.s2 = cur[2];
    qp.pre_n = nxt[0]; qp.s1_n = nxt[1]; qp.s2_n = nxt[2];
    qp.row0 = row0; qp.n_local = n_local; qp.next_row0 = next_row0; qp.out_stored = out_stored ? 1u : 0u;
    const u32 full_w[3] = {prog->pre_width, prog->main_width, prog->stage2_width};
    for (int k = 0; k < 3; k++) {
        qp.wn[k] = next_widths3 ? next_widths3[k] : full_w[k];
        qp.cn[k] = next_col0_3 ? next_col0_3[k] : 0;
    }
    const SelCache& sel = selectors(c, log_n, log_q);
    // alpha powers reversed (src/prover.rs:798-808): constraint j of k weighted by alpha^{k-1-j}
    u32 k = prog->n_zeros + 2 * std::max<u32>(prog->n_lookups, 1);
    std::vector<u64> apow(2 * (size_t)k);
    msh::Fp2 alpha{msh::Fp(alpha2[0]), msh::Fp(alpha2[1])}, acc = msh::Fp2::one();
    for (u32 j = 0; j < k; j++) {
        apow[2 * (size_t)(k - 1 - j)] = acc.c[0].v;
        apow[2 * (size_t)(k - 1 - j) + 1] = acc.c[1].v;
        acc *= alpha;
    }
    DevBuf d_apow(c, apow.size() * 8);
    MSG_CUDA(cudaMemcpyAsync(d_apow.p, apow.data(), apow.size() * 8, cudaMemcpyHostToDevice, c.stream));
    msh::Fp inj_norm = (msh::Fp((msh::u64)n) * msh::two_adic_generator(log_n)).inverse();
    qp.prog = prog->d_full.get();
    qp.n_instr = prog->n_full;
    qp.zero_slots = prog->d_zero_slots.get();
    qp.n_zeros = prog->n_zeros;
    qp.n_lookups = prog->n_lookups;
    qp.lk_mult = prog->d_mult_full.get();
    qp.lk_argoff = prog->d_arg_off.get();
    qp.lk_args = prog->d_args_full.get();
    qp.wpre = prog->pre_width;
    qp.w1 = prog->main_width;
    qp.w2 = prog->stage2_width;
    qp.apow = d_apow.u();
    qp.sel_first = sel.first.get();
    qp.sel_last = sel.last.get();
    qp.inv_zh = sel.inv_zh.get();
    qp.out = out;
    qp.xtab = coset_x_table(c, log_nq);
    for (int i = 0; i < 8; i++) qp.publics[i] = publics8[i];
    qp.delta[0] = ((msh::Fp(publics8[6]) - msh::Fp(publics8[4])) * inj_norm).v;
    qp.delta[1] = ((msh::Fp(publics8[7]) - msh::Fp(publics8[5])) * inj_norm).v;
    qp.g_inv = msh::two_adic_generator(log_n).inverse().v;
    qp.log_nq = log_nq;
    qp.log_q = log_q;
    if (n_local) {
        launch_by_slots(prog->slots_full, [&](auto ns) {
            launch(c, "k_quotient_eval", k_quotient_eval<decltype(ns)::value>, (unsigned)((n_local + 127) / 128), kInterpThreads, 0, qp);
        });
    }
    c.sync();  // apow (pageable) must outlive the copy; also surfaces kernel faults here
}

// quotient evaluations in natural order (nq x 2, device; overwritten) -> LDE of the shifted slices (src/prover.rs:631-717)
static u64* quotient_finish(Ctx& c, u64* qv, u32 log_n, u32 log_q, u32 log_blowup) {
    const u32 log_nq = log_n + log_q;
    const u64 nq = 1ull << log_nq, n = 1ull << log_n, q = 1ull << log_q;
    // shifted_quotient_slices: one DFT of the nq x 2 matrix + gather; then the LDE from coefficients
    ntt_dft_bitrev(c, qv, qv, nq, 2, false);
    DevBuf sl(c, n * q * 16);
    quotient_slices(c, qv, sl.u(), log_nq, log_n, 2);
    DevBuf lde(c, (n << log_blowup) * q * 16);
    ntt_lde_from_coeffs(c, sl.u(), lde.u(), n, 2 * q, log_blowup);
    c.sync();
    return (u64*)lde.release();
}
}  // namespace msg

extern "C" {

int msgpu_quotient(msgpu_ctx* h, const msgpu_program* prog, const msgpu_pdata* pd_pre, uint64_t idx_pre,
                   const msgpu_pdata* pd_s1, uint64_t idx_s1, const msgpu_pdata* pd_s2, uint64_t idx_s2, uint32_t log_n,
                   uint32_t log_q, uint32_t log_blowup, const uint64_t* publics8, const uint64_t* alpha2,
                   uint64_t** lde_out_dev, uint64_t* quotient_values_out) {
    return guard([&] {
        Ctx& c = h->c;
        StageScope ss(c, "quotient");
        MSG_REQUIRE(prog && pd_s1 && pd_s2 && publics8 && alpha2 && lde_out_dev, "quotient: null argument");
        MSG_REQUIRE(log_q <= log_blowup, "quotient: quotient degree exceeds the blowup");
        MSG_REQUIRE(log_n + log_blowup <= 32, "quotient: domain exceeds the two-adicity of the field");
        const u64 nq = 1ull << (log_n + log_q);
        const u64* cur[3] = {nullptr, nullptr, nullptr};
        if (prog->pre_width) {
            MSG_REQUIRE(pd_pre, "quotient: circuit has a preprocessed trace but no preprocessed commitment was given");
            view_of(pd_pre, idx_pre, nq, prog->pre_width, &cur[0]);
        }
        view_of(pd_s1, idx_s1, nq, prog->main_width, &cur[1]);
        view_of(pd_s2, idx_s2, nq, prog->stage2_width, &cur[2]);
        DevBuf qv(c, nq * 16);
        quotient_eval(c, prog, cur, cur, 0, nq, 0, log_n, log_q, publics8, alpha2, qv.u(), false);
        if (quotient_values_out) {
            MSG_CUDA(cudaMemcpyAsync(quotient_values_out, qv.p, nq * 16, cudaMemcpyDeviceToHost, c.stream));
            c.sync();
        }
        *lde_out_dev = (uint64_t*)quotient_finish(c, qv.u(), log_n, log_q, log_blowup);
    });
}

// ---- the quotient stage over ROW SHARDS (one proof over several GPUs) -------------------------------------------------------
// values_shard: this rank's stored rows [row0, row0 + n_local) of the quotient domain (the first n*q stored rows of the committed
// LDEs). cur3 / next3: DEVICE pointers (pre, stage 1, stage 2; pre may be NULL) to the local rows and to the shard that holds
// the rows one trace step further (stored rows from next_row0 on; the caller fetched it from its owner -- for the local shard
// itself pass the cur pointers and row0). out_dev: n_local x 2 quotient evaluations in STORED order.
int msgpu_quotient_values_shard(msgpu_ctx* h, const msgpu_program* prog, const uint64_t* const* cur3, const uint64_t* const* next3,
                                const uint32_t* next_widths3, const uint32_t* next_col0_3, uint64_t row0, uint64_t n_local,
                                uint64_t next_row0, uint32_t log_n, uint32_t log_q, const uint64_t* publics8, const uint64_t* alpha2,
                                uint64_t* out_dev) {
    return guard([&] {
        Ctx& c = h->c;
        StageScope ss(c, "quotient");
        MSG_REQUIRE(prog && cur3 && next3 && publics8 && alpha2 && (out_dev || n_local == 0), "quotient_values_shard: null argument");
        MSG_REQUIRE(log_n + log_q <= 32 && (n_local == 0 || row0 + n_local <= (1ull << (log_n + log_q))),
                    "quotient_values_shard: rows outside the quotient domain");
        MSG_REQUIRE((prog->pre_width == 0 || (cur3[0] && next3[0])) && cur3[1] && cur3[2] && next3[1] && next3[2], "quotient_values_shard: missing matrix");
        const u64* cur[3] = {(const u64*)cur3[0], (const u64*)cur3[1], (const u64*)cur3[2]};
        const u64* nxt[3] = {(const u64*)next3[0], (const u64*)next3[1], (const u64*)next3[2]};
        quotient_eval(c, prog, cur, nxt, row0, n_local, next_row0, log_n, log_q, publics8, alpha2, (u64*)out_dev, true, next_widths3,
                      next_col0_3);
    });
}
// dst[r][c - c0] = src[r][c] for c in [c0, c1): the columns of a shard that another shard reads at its next rows
__global__ void __launch_bounds__(256) k_extract_columns(const u64* src, u64 rows, u32 w, u32 c0, u32 wc, u64* dst) {
    const u64 total = rows * wc;
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (u64)gridDim.x * blockDim.x)
        dst[e] = src[(e / wc) * w + c0 + (u32)(e % wc)];
}
int msgpu_extract_columns_dev(msgpu_ctx* h, const uint64_t* src, uint64_t rows, uint64_t width, uint64_t c0, uint64_t c1, uint64_t* dst) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(src && dst && c0 < c1 && c1 <= width, "extract_columns: bad column range");
        if (rows == 0) return;
        StageScope ss(c, "exchange");
        launch(c, "k_extract_columns", k_extract_columns, (unsigned)std::min<u64>((rows * (c1 - c0) + 255) / 256, (u64)c.sm_count * 16), 256, 0,
               (const u64*)src, rows, (u32)width, (u32)c0, (u32)(c1 - c0), (u64*)dst);
    });
}
// values_stored_dev: ALL nq x 2 quotient evaluations in stored (bit-reversed) order, gathered from the shards (device, not
// modified). Returns the quotient LDE as msgpu_quotient does.
int msgpu_quotient_finish(msgpu_ctx* h, const uint64_t* values_stored_dev, uint32_t log_n, uint32_t log_q, uint32_t log_blowup,
                          uint64_t** lde_out_dev) {
    return guard([&] {
        Ctx& c = h->c;
        StageScope ss(c, "quotient");
        MSG_REQUIRE(values_stored_dev && lde_out_dev && log_q <= log_blowup && log_n + log_blowup <= 32, "quotient_finish: bad argument");
        const u64 nq = 1ull << (log_n + log_q);
        DevBuf qv(c, nq * 16);
        ntt_bit_reverse_rows(c, (const u64*)values_stored_dev, qv.u(), nq, 2);
        *lde_out_dev = (uint64_t*)quotient_finish(c, qv.u(), log_n, log_q, log_blowup);
    });
}

int msgpu_shifted_quotient_slices(msgpu_ctx* h, const uint64_t* in, uint64_t nq, uint64_t d, uint64_t q, uint64_t* out) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(is_pow2(nq) && is_pow2(q) && q <= nq && d > 0, "shifted_quotient_slices: bad shape");
        DevBuf din(c, nq * d * 8), dout(c, nq * d * 8);
        MSG_CUDA(cudaMemcpyAsync(din.p, in, nq * d * 8, cudaMemcpyHostToDevice, c.stream));
        ntt_dft_bitrev(c, din.u(), din.u(), nq, d, false);
        quotient_slices(c, din.u(), dout.u(), ilog2(nq), ilog2(nq / q), (u32)d);
        MSG_CUDA(cudaMemcpyAsync(out, dout.p, nq * d * 8, cudaMemcpyDeviceToHost, c.stream));
        c.sync();
    });
}

// Test hook: the selector tables the quotient kernel reads (`trace_domain.selectors_on_coset(quotient_domain)`,
// src/prover.rs:775), in NATURAL order of the quotient coset: point i is x_i = GENERATOR * w_{nq}^i.
int msgpu_selectors_on_coset(msgpu_ctx* h, uint32_t log_n, uint32_t log_q, uint64_t* is_first_row, uint64_t* is_last_row,
                             uint64_t* inv_vanishing) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(log_n + log_q <= msh::GL_TWO_ADICITY && is_first_row && is_last_row && inv_vanishing, "selectors: bad argument");
        const SelCache& sc = selectors(c, log_n, log_q);
        const u32 log_nq = log_n + log_q;
        const u64 nq = 1ull << log_nq, q = 1ull << log_q;
        std::vector<u64> first(nq), last(nq), izh(q);
        MSG_CUDA(cudaMemcpyAsync(first.data(), sc.first.get(), nq * 8, cudaMemcpyDeviceToHost, c.stream));
        MSG_CUDA(cudaMemcpyAsync(last.data(), sc.last.get(), nq * 8, cudaMemcpyDeviceToHost, c.stream));
        MSG_CUDA(cudaMemcpyAsync(izh.data(), sc.inv_zh.get(), q * 8, cudaMemcpyDeviceToHost, c.stream));
        c.sync();
        for (u64 i = 0; i < nq; i++) {  // the tables are kept in stored (bit-reversed) order
            u64 sidx = msh::reverse_bits_len(i, log_nq);
            is_first_row[i] = first[sidx];
            is_last_row[i] = last[sidx];
            inv_vanishing[i] = izh[i & (q - 1)];
        }
    });
}

}  // extern "C"
