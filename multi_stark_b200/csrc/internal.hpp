// Internal (non-ABI) declarations shared by the .cu translation units of libmsgpu.
#pragma once
#include <chrono>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <tuple>
#include <vector>
#include <stdexcept>

#include <nvtx3/nvToolsExt.h>  // header-only: ranges cost nothing unless a tool (ncu --nvtx, nsys) is attached

#include "gl.cuh"
#include "../host/goldilocks.hpp"

namespace msg {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define MSG_CUDA(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            throw msg::Error(-2, std::string(#expr) + ": " + cudaGetErrorString(_e) + " at " + __FILE__ + ":" + \
                                     std::to_string(__LINE__));                                          \
    } while (0)

#define MSG_REQUIRE(cond, msg_)                                  \
    do {                                                         \
        if (!(cond)) throw msg::Error(-1, std::string(msg_));    \
    } while (0)

// Owner of a cudaMalloc'd table that lives as long as the context (Ctx caches, program uploads)
struct CudaFree {
    void operator()(void* p) const noexcept { cudaFree(p); }
};
template <class T>
using CudaPtr = std::unique_ptr<T, CudaFree>;
template <class T>
CudaPtr<T> cuda_malloc(size_t n) {
    void* p = nullptr;
    MSG_CUDA(cudaMalloc(&p, n * sizeof(T)));
    return CudaPtr<T>((T*)p);
}

struct DevPow {
    CudaPtr<u64> lo, hi;
    u32 h1 = 0;
    gl::PowTable view() const { gl::PowTable t; t.lo = lo.get(); t.hi = hi.get(); t.h1 = h1; return t; }
};

struct Ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;  // lazily created: host-to-device prefetches that overlap kernels of `stream`
    unsigned long long launches = 0;  // kernels of this library launched so far
    bool canonicalize_inputs = false;  // MSGPU_OPT_CANONICALIZE_INPUTS: host matrices are reduced mod p on the device after upload
    int sm_count = 148;
    CudaPtr<u64> tw_full[2];  // w_1024^{i} / w_1024^{-i}, i < 1024
    std::map<std::tuple<u32, u32, u32, u64>, CudaPtr<u64>> ntt_tables;  // per-size inter-pass twiddles / coset scales (ntt.cu)
    std::map<std::tuple<u64, u64, u32>, DevPow> pow_cache;
    std::map<std::tuple<u32, u32, u64>, CudaPtr<gl::PowTable>> coset_cache;  // (log_n, added_bits, shift) -> device array [B]
    struct SelCache {
        CudaPtr<u64> first, last, inv_zh, zh;
    };
    std::map<std::pair<u32, u32>, SelCache> sel_cache;  // selectors on the quotient coset per (log_n, log_q)

    // optional per-launch timing (bench.py roofline): CUDA events on the launching stream
    struct ProfRec {
        const char* stage;
        const char* kernel;
        cudaEvent_t a, b;
        double host_us;  // host clock when the launch was issued (MSGPU_TIMELINE diagnostics)
    };
    bool profiling = false;
    const char* stage = "";
    std::vector<ProfRec> prof;

    // Device memory: a caching arena over cudaMalloc'd segments. Every launch and copy of a context goes to its one stream, so
    // a block freed on the host can be handed out again at once (the next user is ordered behind the previous one on the
    // stream). Steady-state proving therefore makes no driver allocation calls at all: cudaMallocAsync / cudaFreeAsync cost
    // up to several ms per large block on a busy box (tools/diag_step.py), more than the kernels they feed.
    struct Arena {
        struct Block {
            size_t size;
            bool free;
            size_t segment;
        };
        std::map<char*, Block> blocks;                 // every block of every segment, by address
        std::multimap<size_t, char*> free_by_size;     // free blocks
        std::vector<std::pair<char*, size_t>> segments;
        size_t reserved = 0, in_use = 0, peak_in_use = 0;
    } arena;
    Ctx() = default;
    ~Ctx();  // synchronises the stream, then frees the tables, the arena and the streams this context created
    void* alloc(size_t bytes);  // valid for work enqueued on `stream` after the call
    bool free(void* p) noexcept;  // the block may be reused by later work on `stream`; false = not a live block
    void arena_trim();          // give wholly free segments back to the driver
    void arena_destroy();
    void sync() { MSG_CUDA(cudaStreamSynchronize(stream)); }
    const DevPow& pow_table(u64 g, u64 c, u32 bits);
    const gl::PowTable* coset_tables(u32 log_n, u32 added_bits, u64 shift);
    const gl::PowTable* lde_coeff_tables(u32 log_n, u32 added_bits);
};

void ctx_init_tables(Ctx& c);

// Opt a kernel in to more than 48 KB of dynamic shared memory, once per (device, kernel): the attribute belongs to the
// device's instance of the function, so a process-wide "done" flag would leave a second device without it.
template <class F>
inline void ensure_max_smem(F* func, int bytes) {
    static std::mutex mu;
    static std::set<std::pair<int, const void*>> done;
    int dev = 0;
    MSG_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    if (done.count({dev, (const void*)func})) return;
    MSG_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    done.insert({dev, (const void*)func});
}

// Owner of one arena block of a context (Ctx::alloc). Empty when default-constructed, moved from or released.
struct DevBuf {
    Ctx* c = nullptr;
    void* p = nullptr;
    DevBuf() = default;
    DevBuf(Ctx& c_, size_t bytes) : c(&c_), p(c_.alloc(bytes)) {}
    DevBuf(Ctx& c_, void* adopted) : c(&c_), p(adopted) {}  // takes over a live block of c_ (msgpu_malloc)
    DevBuf(DevBuf&& o) noexcept : c(o.c), p(o.release()) {}
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) {
            reset();
            c = o.c;
            p = o.release();
        }
        return *this;
    }
    ~DevBuf() { reset(); }
    void reset() noexcept {
        if (p) c->free(p);
        p = nullptr;
    }
    void* release() noexcept {
        void* r = p;
        p = nullptr;
        return r;
    }
    explicit operator bool() const { return p != nullptr; }
    u64* u() const { return (u64*)p; }
    uint8_t* bytes() const { return (uint8_t*)p; }
};

// Owner of the event that marks the end of a copy into an arena block. It waits for the event before destroying it: a copy must
// not outlive its block, so the owner is declared after the block's DevBuf (members are destroyed in reverse order).
struct Event {
    cudaEvent_t e = nullptr;
    Event() = default;
    Event(Event&& o) noexcept : e(o.e) { o.e = nullptr; }
    Event& operator=(Event&&) = delete;
    ~Event() {
        if (e) {
            cudaEventSynchronize(e);
            cudaEventDestroy(e);
        }
    }
    void record(cudaStream_t s) {
        if (!e) MSG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        MSG_CUDA(cudaEventRecord(e, s));
    }
};

inline double host_now_us() {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
// Every kernel of this library is launched here, on the context's stream: the launch is counted, timed under `name` when
// profiling (bench.py looks kernels up by these names) and checked.
template <class... P, class... A>
void launch(Ctx& c, const char* name, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, A&&... args) {
    cudaEvent_t b = nullptr;
    if (c.profiling) {
        cudaEvent_t a;
        MSG_CUDA(cudaEventCreate(&a));
        MSG_CUDA(cudaEventCreate(&b));
        MSG_CUDA(cudaEventRecord(a, c.stream));
        c.prof.push_back(Ctx::ProfRec{c.stage, name, a, b, host_now_us()});
    }
    kernel<<<grid, block, smem, c.stream>>>(std::forward<A>(args)...);
    c.launches++;
    if (b) cudaEventRecord(b, c.stream);
    MSG_CUDA(cudaGetLastError());
}
// Names the stage of the launches inside it: the per-launch profile of bench.py groups by it, and it is an NVTX range named
// after the reference's tracing spans (SURVEY 5: "stark/stage1_commit" ... are spans of src/prover.rs; the stages here are
// the device-side pieces of those spans: lde, merkle, stage2, quotient, open, fri, transcript, exchange), so that
// `ncu --nvtx --nvtx-include "lde/"` or an nsys timeline shows the same structure.
struct StageScope {
    Ctx& c;
    const char* prev;
    StageScope(Ctx& c_, const char* s) : c(c_), prev(c_.stage) {
        c.stage = s;
        nvtxRangePushA(s);
    }
    ~StageScope() {
        c.stage = prev;
        nvtxRangePop();
    }
};

// ---- NTT / LDE (ntt.cu) -------------------------------------------------------------------
// Forward (or inverse, unnormalised) DFT of every column; natural order in, bit-reversed rows out.
void ntt_dft_bitrev(Ctx& c, const u64* src, u64* dst, u64 n, u64 w, bool inverse, u64 batch = 1);
// coset_lde_batch(evals, added_bits, shift).bit_reverse_rows(); tmp holds n*w elements.
void ntt_coset_lde(Ctx& c, const u64* src, u64* dst, u64* tmp, u64 n, u64 w, u32 added_bits, u64 shift);
// zero-pad coefficient rows to n << added_bits, one DFT, bit-reversed rows (src/prover.rs:709-717)
void ntt_lde_from_coeffs(Ctx& c, const u64* src, u64* dst, u64 n, u64 w, u32 added_bits);
// natural-order inverse DFT (with 1/n); tmp holds n*w elements
void ntt_idft_natural(Ctx& c, const u64* src, u64* dst, u64* tmp, u64 n, u64 w);
// dst[r] = src[rev(r)]
void ntt_bit_reverse_rows(Ctx& c, const u64* src, u64* dst, u64 n, u64 w);

// ---- BLAKE3 Merkle (merkle.cu) ------------------------------------------------------------------
struct MatRef {
    const u64* ptr;
    u64 height;
    u64 width;
};
// mats[first .. first + count) are the column blocks (dense height x width_b, in column order) of ONE matrix that the leaf pass
// also writes out, row-major over all its columns, to dst
struct AsmTarget {
    size_t first, count;
    u64* dst;
};
// digests[i] = BLAKE3(le_bytes(row i of mats[0]) || le_bytes(row i of mats[1]) ...), all mats same height
void b3_hash_rows(Ctx& c, const std::vector<MatRef>& mats, uint8_t* digests, const std::vector<AsmTarget>& assemble = {});
// next[i] = H(prev[2i] || prev[2i+1]), optionally followed by H(that || inject[i])
void b3_compress_layer(Ctx& c, const uint8_t* prev, const uint8_t* inject, uint8_t* next, u64 next_len);

// `levels` node layers in one launch (each CTA reduces 2^levels adjacent digests through shared memory)
void b3_merkle_subtrees(Ctx& c, const uint8_t* in, u64 len, u32 levels, uint8_t* const* out, const uint8_t* const* inject);
// BLAKE3 of one long (> 1024 bytes) device-resident byte string; out_dev receives 32 bytes
void b3_hash_long(Ctx& c, const uint8_t* data_dev, u64 len, uint8_t* out_dev);
// sets *flag_dev |= 1 if any v[i] >= p
void check_canonical(Ctx& c, const u64* v, u64 n, u32* flag_dev);
// v[i] <- v[i] mod p in place (device)
void canonicalize(Ctx& c, u64* v, u64 n);

inline unsigned ilog2(u64 n) {
    unsigned l = 0;
    while ((1ull << l) < n) l++;
    return l;
}
inline bool is_pow2(u64 n) { return n && !(n & (n - 1)); }

}  // namespace msg
