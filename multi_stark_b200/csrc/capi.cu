// extern "C" surface of libmsgpu (include/msgpu.h). Every entry point catches C++ exceptions and
// turns them into error codes + a thread-local message; nothing unwinds across the ABI.
#include "capi_common.hpp"
#include "mmcs.hpp"
#include "../host/blake3_host.hpp"
#include <algorithm>
#include <cstring>
#include <iterator>

namespace msg {

static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }

static constexpr size_t kArenaAlign = 512;            // keeps 128-bit vector accesses and TMA-sized rows aligned
static constexpr size_t kArenaMinSegment = 64u << 20;  // small requests share 64 MB segments

static void arena_erase_free(Ctx::Arena& a, char* addr, size_t size) {
    auto range = a.free_by_size.equal_range(size);
    for (auto it = range.first; it != range.second; ++it)
        if (it->second == addr) {
            a.free_by_size.erase(it);
            return;
        }
}

void* Ctx::alloc(size_t bytes) {
    Arena& a = arena;
    size_t need = ((bytes ? bytes : 8) + kArenaAlign - 1) / kArenaAlign * kArenaAlign;
    auto fit = a.free_by_size.lower_bound(need);
    if (fit == a.free_by_size.end()) {
        // no block fits: a new segment, exactly the request for large blocks (a proof repeats its sizes)
        size_t seg = need >= kArenaMinSegment ? (need + (2u << 20) - 1) / (2u << 20) * (2u << 20) : kArenaMinSegment;
        void* base = nullptr;
        cudaError_t e = cudaMalloc(&base, seg);
        if (e != cudaSuccess) {
            cudaGetLastError();
            MSG_CUDA(cudaStreamSynchronize(stream));
            arena_trim();
            e = cudaMalloc(&base, seg);
        }
        if (e != cudaSuccess) {
            cudaGetLastError();
            throw Error(MSGPU_ERR_CUDA, "out of device memory: " + std::to_string(seg >> 20) + " MB requested, " +
                                            std::to_string(a.reserved >> 20) + " MB reserved, " + std::to_string(a.in_use >> 20) + " MB in use");
        }
        a.segments.push_back({(char*)base, seg});
        a.reserved += seg;
        a.blocks[(char*)base] = Arena::Block{seg, true, a.segments.size() - 1};
        fit = a.free_by_size.insert({seg, (char*)base});
    }
    char* addr = fit->second;
    a.free_by_size.erase(fit);
    Arena::Block& b = a.blocks[addr];
    if (b.size - need >= kArenaAlign) {  // split: the tail stays free
        char* tail = addr + need;
        a.blocks[tail] = Arena::Block{b.size - need, true, b.segment};
        a.free_by_size.insert({b.size - need, tail});
        b.size = need;
    }
    b.free = false;
    a.in_use += b.size;
    a.peak_in_use = std::max(a.peak_in_use, a.in_use);
    return addr;
}

bool Ctx::free(void* p) noexcept {
    if (!p) return true;
    Arena& a = arena;
    auto it = a.blocks.find((char*)p);
    if (it == a.blocks.end() || it->second.free) return false;  // not a live block of this context
    it->second.free = true;
    a.in_use -= it->second.size;
    // merge with the free neighbours of the same segment
    auto nxt = std::next(it);
    if (nxt != a.blocks.end() && nxt->second.free && nxt->second.segment == it->second.segment && it->first + it->second.size == nxt->first) {
        arena_erase_free(a, nxt->first, nxt->second.size);
        it->second.size += nxt->second.size;
        a.blocks.erase(nxt);
    }
    if (it != a.blocks.begin()) {
        auto prv = std::prev(it);
        if (prv->second.free && prv->second.segment == it->second.segment && prv->first + prv->second.size == it->first) {
            arena_erase_free(a, prv->first, prv->second.size);
            prv->second.size += it->second.size;
            a.blocks.erase(it);
            it = prv;
        }
    }
    a.free_by_size.insert({it->second.size, it->first});
    return true;
}

void Ctx::arena_trim() {
    Arena& a = arena;
    for (size_t s = 0; s < a.segments.size(); s++) {
        char* base = a.segments[s].first;
        if (!base) continue;
        auto it = a.blocks.find(base);
        if (it == a.blocks.end() || !it->second.free || it->second.size != a.segments[s].second) continue;
        arena_erase_free(a, base, it->second.size);
        a.blocks.erase(it);
        cudaFree(base);
        a.reserved -= a.segments[s].second;
        a.segments[s] = {nullptr, 0};
    }
}

void Ctx::arena_destroy() {
    for (auto& s : arena.segments)
        if (s.first) cudaFree(s.first);
    arena = Arena();
}

Ctx::~Ctx() {
    cudaSetDevice(device);
    if (stream) cudaStreamSynchronize(stream);
    for (auto& t : tw_full) t.reset();
    ntt_tables.clear();
    pow_cache.clear();
    coset_cache.clear();
    sel_cache.clear();
    arena_destroy();
    if (copy_stream) cudaStreamDestroy(copy_stream);
    if (own_stream) cudaStreamDestroy(stream);
}

void b3_compress_raw_dev(Ctx& c, const u32* st, const u32* msg, u32* out);

static void check_shape(u64 rows, u64 cols) {
    MSG_REQUIRE(is_pow2(rows), "matrix height must be a power of two");
    MSG_REQUIRE(cols == 0 || rows <= (~0ull) / 8 / cols, "matrix too large");
}

// shared body of the host-pointer DFT entry points: upload, run, download
template <class F>
static void host_transform(Ctx& c, const u64* in, u64 rows, u64 cols, u64 out_rows, u64* out, F&& run) {
    check_shape(rows, cols);
    if (rows * cols == 0) return;
    DevBuf din(c, rows * cols * 8), dout(c, out_rows * cols * 8);
    MSG_CUDA(cudaMemcpyAsync(din.p, in, rows * cols * 8, cudaMemcpyHostToDevice, c.stream));
    run(din.u(), dout.u());
    MSG_CUDA(cudaMemcpyAsync(out, dout.p, out_rows * cols * 8, cudaMemcpyDeviceToHost, c.stream));
    c.sync();
}

static std::unique_ptr<msgpu_pdata> commit_impl(Ctx& c, const u64* const* mats, const u64* heights, const u64* widths, u64 n,
                                                u32 log_blowup, bool host_inputs, bool do_lde) {
    MSG_REQUIRE(n > 0, "commit: no matrices given");
    auto pd = std::make_unique<msgpu_pdata>();
    for (u64 i = 0; i < n; i++) {
        check_shape(heights[i], widths[i]);
        u64 h = heights[i], w = widths[i];
        pd->mats.push_back(msgpu_pdata::Mat::alloc(c, do_lde ? (h << log_blowup) : h, w));
        u64* out = pd->mats.back().ptr;
        if (w == 0) continue;
        if (!do_lde) {
            MSG_CUDA(cudaMemcpyAsync(out, mats[i], h * w * 8, host_inputs ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, c.stream));
            continue;
        }
        StageScope stage_scope(c, "lde");
        DevBuf tmp(c, h * w * 8);
        if (host_inputs) {
            MSG_CUDA(cudaMemcpyAsync(tmp.p, mats[i], h * w * 8, cudaMemcpyHostToDevice, c.stream));
            if (c.canonicalize_inputs) canonicalize(c, tmp.u(), h * w);
            ntt_coset_lde(c, tmp.u(), out, tmp.u(), h, w, log_blowup, msh::GL_GENERATOR);
        } else {
            ntt_coset_lde(c, mats[i], out, tmp.u(), h, w, log_blowup, msh::GL_GENERATOR);
        }
    }
    mmcs_build(c, pd.get());
    return pd;
}

}  // namespace msg

using namespace msg;

extern "C" {

int msgpu_ctx_create(int device, void* stream, msgpu_ctx** out) {
    return guard([&] {
        MSG_REQUIRE(out != nullptr, "ctx_create: null output");
        int count = 0;
        MSG_CUDA(cudaGetDeviceCount(&count));
        MSG_REQUIRE(device >= 0 && device < count, "ctx_create: no such CUDA device (libmsgpu has no CPU fallback)");
        MSG_CUDA(cudaSetDevice(device));
        auto h = std::make_unique<msgpu_ctx>();
        h->c.device = device;
        if (stream) {
            h->c.stream = (cudaStream_t)stream;
        } else {
            MSG_CUDA(cudaStreamCreateWithFlags(&h->c.stream, cudaStreamNonBlocking));
            h->c.own_stream = true;
        }
        cudaDeviceProp prop;
        MSG_CUDA(cudaGetDeviceProperties(&prop, device));
        h->c.sm_count = prop.multiProcessorCount;
        ctx_init_tables(h->c);
        *out = h.release();
    });
}

void msgpu_ctx_destroy(msgpu_ctx* h) { delete h; }

const char* msgpu_last_error(void) { return g_last_error.c_str(); }
int msgpu_sync(msgpu_ctx* h) {
    return guard([&] { h->c.sync(); });
}
void* msgpu_stream(msgpu_ctx* h) { return (void*)h->c.stream; }
uint64_t msgpu_launch_count(msgpu_ctx* h) { return h->c.launches; }

int msgpu_malloc(msgpu_ctx* h, size_t bytes, void** dptr) {
    return guard([&] { *dptr = h->c.alloc(bytes); });
}
int msgpu_free(msgpu_ctx* h, void* dptr) {
    return guard([&] { MSG_REQUIRE(h->c.free(dptr), "free: not a live block of this context"); });
}
int msgpu_arena_in_use(msgpu_ctx* h, uint64_t* bytes) {
    return guard([&] {
        MSG_REQUIRE(h && bytes, "arena_in_use: null argument");
        *bytes = h->c.arena.in_use;
    });
}
int msgpu_memcpy_h2d(msgpu_ctx* h, void* dst, const void* src, size_t bytes) {
    return guard([&] {
        MSG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->c.stream));
        h->c.sync();
    });
}
int msgpu_memcpy_d2h(msgpu_ctx* h, void* dst, const void* src, size_t bytes) {
    return guard([&] {
        MSG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->c.stream));
        h->c.sync();
    });
}
int msgpu_host_alloc(size_t bytes, void** hptr) {
    return guard([&] { MSG_CUDA(cudaHostAlloc(hptr, bytes ? bytes : 8, cudaHostAllocDefault)); });
}
int msgpu_host_free(void* hptr) {
    return guard([&] { MSG_CUDA(cudaFreeHost(hptr)); });
}
// Page-lock memory the caller already owns (a `RowMajorMatrix<Goldilocks>`'s Vec): the host-pointer entry points then copy
// straight from it at full PCIe rate, with no staging copy on either side.
int msgpu_host_register(void* hptr, size_t bytes) {
    return guard([&] {
        MSG_REQUIRE(hptr && bytes, "host_register: null or empty range");
        MSG_CUDA(cudaHostRegister(hptr, bytes, cudaHostRegisterDefault));
    });
}
int msgpu_host_unregister(void* hptr) {
    return guard([&] { MSG_CUDA(cudaHostUnregister(hptr)); });
}
int msgpu_ctx_set_option(msgpu_ctx* h, int option, uint64_t value) {
    return guard([&] {
        MSG_REQUIRE(h, "ctx_set_option: null context");
        switch (option) {
            case MSGPU_OPT_CANONICALIZE_INPUTS: h->c.canonicalize_inputs = value != 0; break;
            default: throw Error(-1, "ctx_set_option: unknown option");
        }
    });
}

int msgpu_upload_canonical(msgpu_ctx* h, void* dst, const uint64_t* src, uint64_t n) {
    return guard([&] {
        Ctx& c = h->c;
        if (n == 0) return;
        MSG_CUDA(cudaMemcpyAsync(dst, src, n * 8, cudaMemcpyHostToDevice, c.stream));
        if (c.canonicalize_inputs) {
            canonicalize(c, (u64*)dst, n);
            c.sync();
            return;
        }
        DevBuf flag(c, 4);
        MSG_CUDA(cudaMemsetAsync(flag.p, 0, 4, c.stream));
        check_canonical(c, (const u64*)dst, n, (u32*)flag.p);
        u32 bad = 0;
        MSG_CUDA(cudaMemcpyAsync(&bad, flag.p, 4, cudaMemcpyDeviceToHost, c.stream));
        c.sync();
        MSG_REQUIRE(bad == 0, "upload: value is not a canonical field element (>= p)");
    });
}

int msgpu_blake3_hash(msgpu_ctx* h, const uint8_t* data, uint64_t len, uint8_t* out32) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(out32 && (data || len == 0), "blake3_hash: null argument");
        if (len <= 1024) {  // a single chunk: not worth a launch
            msh::Digest d = msh::blake3_hash(data, (size_t)len);
            memcpy(out32, d.data(), 32);
            return;
        }
        StageScope ss(c, "transcript");
        DevBuf buf(c, len + 64);
        uint8_t* out_dev = (uint8_t*)buf.p + ((len + 15) / 16) * 16;
        MSG_CUDA(cudaMemcpyAsync(buf.p, data, len, cudaMemcpyHostToDevice, c.stream));
        b3_hash_long(c, (const uint8_t*)buf.p, len, out_dev);
        MSG_CUDA(cudaMemcpyAsync(out32, out_dev, 32, cudaMemcpyDeviceToHost, c.stream));
        c.sync();
    });
}

int msgpu_profile_begin(msgpu_ctx* h) {
    return guard([&] {
        Ctx& c = h->c;
        for (auto& r : c.prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        c.prof.clear();
        c.profiling = true;
    });
}
int msgpu_profile_end(msgpu_ctx* h, char* json_out, size_t cap) {
    return guard([&] {
        Ctx& c = h->c;
        c.profiling = false;
        c.sync();
        // aggregate by (stage, kernel)
        std::map<std::pair<std::string, std::string>, std::pair<double, unsigned long long>> agg;
        std::vector<std::pair<std::string, std::string>> order;
        const bool timeline = getenv("MSGPU_TIMELINE") != nullptr;  // diagnostics: one line per launch on stderr
        for (auto& r : c.prof) {
            float ms = 0;
            MSG_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
            if (timeline) {
                float off = 0;
                cudaEventElapsedTime(&off, c.prof.front().a, r.a);
                fprintf(stderr, "[timeline] %-9s %-24s host +%9.1f us  gpu +%9.1f us  dur %8.1f us\n", r.stage, r.kernel,
                        r.host_us - c.prof.front().host_us, off * 1e3, ms * 1e3);
            }
            auto key = std::make_pair(std::string(r.stage), std::string(r.kernel));
            if (!agg.count(key)) order.push_back(key);
            agg[key].first += ms;
            agg[key].second += 1;
        }
        for (auto& r : c.prof) {
            cudaEventDestroy(r.a);
            cudaEventDestroy(r.b);
        }
        c.prof.clear();
        std::string js = "[";
        for (size_t i = 0; i < order.size(); i++) {
            auto& v = agg[order[i]];
            char buf[256];
            snprintf(buf, sizeof buf, "%s{\"stage\": \"%s\", \"kernel\": \"%s\", \"launches\": %llu, \"ms\": %.6f}",
                     i ? ", " : "", order[i].first.c_str(), order[i].second.c_str(), v.second, v.first);
            js += buf;
        }
        js += "]";
        MSG_REQUIRE(json_out && js.size() + 1 <= cap, "profile_end: output buffer too small");
        memcpy(json_out, js.c_str(), js.size() + 1);
    });
}

// ---- DFT slot -----------------------------------------------------------------------------------
int msgpu_dft_batch_bitrev(msgpu_ctx* h, const uint64_t* in, uint64_t rows, uint64_t cols, uint64_t* out) {
    return guard([&] {
        Ctx& c = h->c;
        host_transform(c, (const u64*)in, rows, cols, rows, (u64*)out,
                       [&](u64* di, u64* dout) { ntt_dft_bitrev(c, di, dout, rows, cols, false); });
    });
}
int msgpu_dft_batch(msgpu_ctx* h, const uint64_t* in, uint64_t rows, uint64_t cols, uint64_t* out) {
    return guard([&] {
        Ctx& c = h->c;
        host_transform(c, (const u64*)in, rows, cols, rows, (u64*)out, [&](u64* di, u64* dout) {
            ntt_dft_bitrev(c, di, di, rows, cols, false);
            ntt_bit_reverse_rows(c, di, dout, rows, cols);
        });
    });
}
int msgpu_idft_batch(msgpu_ctx* h, const uint64_t* in, uint64_t rows, uint64_t cols, uint64_t* out) {
    return guard([&] {
        Ctx& c = h->c;
        host_transform(c, (const u64*)in, rows, cols, rows, (u64*)out,
                       [&](u64* di, u64* dout) { ntt_idft_natural(c, di, dout, di, rows, cols); });
    });
}
int msgpu_coset_lde_batch_bitrev(msgpu_ctx* h, const uint64_t* in, uint64_t rows, uint64_t cols, uint32_t added_bits,
                                 uint64_t shift, uint64_t* out) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(shift != 0 && shift < GLD_P, "coset_lde: shift must be a non-zero canonical field element");
        MSG_REQUIRE(added_bits <= 32, "coset_lde: added_bits too large");
        host_transform(c, (const u64*)in, rows, cols, rows << added_bits, (u64*)out,
                       [&](u64* di, u64* dout) { ntt_coset_lde(c, di, dout, di, rows, cols, added_bits, shift); });
    });
}
int msgpu_lde_from_shifted_coefficients(msgpu_ctx* h, const uint64_t* in, uint64_t rows, uint64_t cols,
                                        uint32_t added_bits, uint64_t* out) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(added_bits <= 32, "lde: added_bits too large");
        host_transform(c, (const u64*)in, rows, cols, rows << added_bits, (u64*)out,
                       [&](u64* di, u64* dout) { ntt_lde_from_coeffs(c, di, dout, rows, cols, added_bits); });
    });
}
int msgpu_dft_batch_bitrev_dev(msgpu_ctx* h, const uint64_t* in, uint64_t rows, uint64_t cols, uint64_t* out) {
    return guard([&] {
        check_shape(rows, cols);
        ntt_dft_bitrev(h->c, (const u64*)in, (u64*)out, rows, cols, false);
    });
}
int msgpu_coset_lde_batch_bitrev_dev(msgpu_ctx* h, const uint64_t* in, uint64_t rows, uint64_t cols,
                                     uint32_t added_bits, uint64_t shift, uint64_t* out) {
    return guard([&] {
        Ctx& c = h->c;
        check_shape(rows, cols);
        MSG_REQUIRE(shift != 0 && shift < GLD_P, "coset_lde: shift must be a non-zero canonical field element");
        if (rows * cols == 0) return;
        DevBuf tmp(c, rows * cols * 8);
        ntt_coset_lde(c, (const u64*)in, (u64*)out, tmp.u(), rows, cols, added_bits, shift);
    });
}
int msgpu_lde_from_shifted_coefficients_dev(msgpu_ctx* h, const uint64_t* in, uint64_t rows, uint64_t cols,
                                            uint32_t added_bits, uint64_t* out) {
    return guard([&] {
        check_shape(rows, cols);
        ntt_lde_from_coeffs(h->c, (const u64*)in, (u64*)out, rows, cols, added_bits);
    });
}

// ---- PCS / MMCS slot ------------------------------------------------------------------------------
int msgpu_commit(msgpu_ctx* h, const uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths,
                 uint64_t n_mats, uint32_t log_blowup, msgpu_pdata** out, uint8_t* root32) {
    return guard([&] {
        auto pd = commit_impl(h->c, (const u64* const*)mats, (const u64*)heights, (const u64*)widths, n_mats, log_blowup, true, true);
        memcpy(root32, pd->root, 32);
        *out = pd.release();
    });
}
// ---- pipelined host commit: uploads on the copy stream, LDEs on the main stream --------------------------------------------
struct msgpu_upload {
    Ctx* ctx;
    struct Item {
        DevBuf dev;
        u64 height, width;
        Event ready;  // the copy into `dev` has finished
    };
    std::vector<Item> items;
};
int msgpu_upload_begin(msgpu_ctx* h, const uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths, uint64_t n_mats,
                       msgpu_upload** out) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(out && mats && heights && widths && n_mats > 0, "upload_begin: null or empty argument");
        if (!c.copy_stream) MSG_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
        auto up = std::make_unique<msgpu_upload>();
        up->ctx = &c;
        up->items.reserve(n_mats);
        // the blocks may just have been freed by work still running on the main stream: the copies start behind it
        cudaEvent_t e0;
        MSG_CUDA(cudaEventCreateWithFlags(&e0, cudaEventDisableTiming));
        MSG_CUDA(cudaEventRecord(e0, c.stream));
        MSG_CUDA(cudaStreamWaitEvent(c.copy_stream, e0, 0));
        cudaEventDestroy(e0);
        for (u64 i = 0; i < n_mats; i++) {
            check_shape(heights[i], widths[i]);
            const u64 bytes = heights[i] * widths[i] * 8;
            up->items.push_back(msgpu_upload::Item{DevBuf(c, bytes), heights[i], widths[i], Event()});
            auto& it = up->items.back();
            if (bytes) {
                MSG_REQUIRE(mats[i], "upload_begin: null matrix");
                MSG_CUDA(cudaMemcpyAsync(it.dev.p, mats[i], bytes, cudaMemcpyHostToDevice, c.copy_stream));
            }
            it.ready.record(c.copy_stream);
        }
        *out = up.release();
    });
}
void msgpu_upload_free(msgpu_upload* up) { delete up; }
int msgpu_commit_upload(msgpu_upload* up, uint32_t log_blowup, int verify_canonical, uint64_t** kept_inputs, int local_only,
                        msgpu_pdata** out, uint8_t* root32) {
    return guard([&] {
        MSG_REQUIRE(up && out && (root32 || local_only), "commit_upload: null argument");
        std::unique_ptr<msgpu_upload> consumed(up);
        Ctx& c = *up->ctx;
        auto pd = std::make_unique<msgpu_pdata>();
        DevBuf flag(c, 4);
        MSG_CUDA(cudaMemsetAsync(flag.p, 0, 4, c.stream));
        for (auto& it : up->items) {
            // matrix i is extended while matrices i + 1 ... are still arriving
            MSG_CUDA(cudaStreamWaitEvent(c.stream, it.ready.e, 0));
            pd->mats.push_back(msgpu_pdata::Mat::alloc(c, it.height << log_blowup, it.width));
            if (it.width == 0) continue;
            if (c.canonicalize_inputs) canonicalize(c, it.dev.u(), it.height * it.width);
            else if (verify_canonical) check_canonical(c, it.dev.u(), it.height * it.width, (u32*)flag.p);
            StageScope stage_scope(c, "lde");
            DevBuf tmp(c, it.height * it.width * 8);
            ntt_coset_lde(c, it.dev.u(), pd->mats.back().ptr, tmp.u(), it.height, it.width, log_blowup, msh::GL_GENERATOR);
        }
        u32 bad = 0;
        MSG_CUDA(cudaMemcpyAsync(&bad, flag.p, 4, cudaMemcpyDeviceToHost, c.stream));
        if (local_only) {
            mmcs_build_local(c, pd.get());  // leaf digests per height class only (sharded commitments)
            c.sync();
        } else {
            mmcs_build(c, pd.get());  // synchronises
        }
        MSG_REQUIRE(bad == 0, "commit_upload: value is not a canonical field element (>= p)");
        if (kept_inputs)
            for (size_t i = 0; i < up->items.size(); i++) kept_inputs[i] = (uint64_t*)up->items[i].dev.release();
        if (root32) memcpy(root32, pd->root, 32);
        *out = pd.release();
    });
}

int msgpu_commit_dev(msgpu_ctx* h, const uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths,
                     uint64_t n_mats, uint32_t log_blowup, msgpu_pdata** out, uint8_t* root32) {
    return guard([&] {
        auto pd = commit_impl(h->c, (const u64* const*)mats, (const u64*)heights, (const u64*)widths, n_mats, log_blowup, false, true);
        memcpy(root32, pd->root, 32);
        *out = pd.release();
    });
}
// ---- sharded commitments: one MMCS whose matrices live on several GPUs --------------------------------------------------
int msgpu_commit_local_dev(msgpu_ctx* h, uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths, uint64_t n_mats,
                           uint32_t log_blowup, int inputs_are_ldes, msgpu_pdata** out) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(n_mats > 0 && out, "commit_local: no matrices given");
        auto pd = std::make_unique<msgpu_pdata>();
        for (u64 i = 0; i < n_mats; i++) {
            check_shape(heights[i], widths[i]);
            if (inputs_are_ldes) {  // adopted (buffers from msgpu_malloc), as msgpu_commit_ldes_dev with take_ownership = 1
                pd->mats.push_back(msgpu_pdata::Mat{(u64*)mats[i], heights[i], widths[i]});
                continue;
            }
            u64 hh = heights[i], w = widths[i];
            pd->mats.push_back(msgpu_pdata::Mat::alloc(c, hh << log_blowup, w));
            if (w == 0) continue;
            StageScope stage_scope(c, "lde");
            DevBuf tmp(c, hh * w * 8);
            ntt_coset_lde(c, (const u64*)mats[i], pd->mats.back().ptr, tmp.u(), hh, w, log_blowup, msh::GL_GENERATOR);
        }
        mmcs_build_local(c, pd.get());
        // The class digests are handed to the caller's transport next (an NCCL send ordered against ITS stream, not this
        // context's): they must be complete when this call returns, as in the local_only branch of msgpu_commit_upload.
        c.sync();
        if (inputs_are_ldes)
            for (auto& m : pd->mats) m.own = DevBuf(c, (void*)m.ptr);
        *out = pd.release();
    });
}
uint64_t msgpu_pdata_num_classes(const msgpu_pdata* pd) { return pd->class_leaves.size(); }
int msgpu_pdata_class_digests(const msgpu_pdata* pd, uint64_t k, uint64_t* lde_height, uint8_t** dev_ptr) {
    return guard([&] {
        MSG_REQUIRE(k < pd->class_leaves.size(), "class_digests: no such height class");
        if (lde_height) *lde_height = pd->class_leaves[k].first;
        if (dev_ptr) *dev_ptr = pd->class_leaves[k].second.bytes();
    });
}
int msgpu_tree_from_digests(msgpu_ctx* h, uint64_t n_classes, const uint64_t* lde_heights, const uint8_t* const* digests_dev,
                            msgpu_pdata** out, uint8_t* root32) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(n_classes > 0 && lde_heights && digests_dev && out && root32, "tree_from_digests: null argument");
        std::vector<std::pair<u64, const uint8_t*>> classes;
        for (u64 k = 0; k < n_classes; k++) classes.push_back({lde_heights[k], digests_dev[k]});
        std::sort(classes.begin(), classes.end(), [](auto& a, auto& b) { return a.first > b.first; });
        auto pd = std::make_unique<msgpu_pdata>();
        mmcs_build_from_classes(c, pd.get(), classes);
        memcpy(root32, pd->root, 32);
        *out = pd.release();
    });
}
uint64_t msgpu_pdata_max_height(const msgpu_pdata* pd) { return pd->max_height; }
int msgpu_pdata_digests(const msgpu_pdata* pd, uint8_t** dev_ptr, uint64_t* n_digests) {
    return guard([&] {
        MSG_REQUIRE(pd && pd->digests && dev_ptr && n_digests, "pdata_digests: prover data without a tree");
        *dev_ptr = pd->digests.bytes();
        *n_digests = 2 * pd->max_height - 1;
    });
}
int msgpu_pack_column_blocks_dev(msgpu_ctx* h, const uint64_t* src, uint64_t rows, uint64_t width, uint64_t n_blocks, const uint64_t* c0,
                                 const uint64_t* c1, uint64_t* dst) {
    return guard([&] {
        MSG_REQUIRE(src && dst && c0 && c1, "pack_column_blocks: null argument");
        std::vector<u64*> blocks;
        for (u64 b = 0; b < n_blocks; b++) blocks.push_back((u64*)dst + rows * c0[b]);
        StageScope ss(h->c, "exchange");
        pack_column_blocks(h->c, (const u64*)src, rows, width, std::vector<u64>(c0, c0 + n_blocks), std::vector<u64>(c1, c1 + n_blocks), blocks);
    });
}
int msgpu_interleave_column_blocks_dev(msgpu_ctx* h, const uint64_t* src, uint64_t rows, uint64_t n_blocks, const uint64_t* widths,
                                       uint64_t* dst) {
    return guard([&] {
        MSG_REQUIRE(src && dst && widths, "interleave_column_blocks: null argument");
        StageScope ss(h->c, "exchange");
        interleave_column_blocks(h->c, (const u64*)src, rows, std::vector<u64>(widths, widths + n_blocks), (u64*)dst);
    });
}

int msgpu_mmcs_commit(msgpu_ctx* h, const uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths,
                      uint64_t n_mats, msgpu_pdata** out, uint8_t* root32) {
    return guard([&] {
        auto pd = commit_impl(h->c, (const u64* const*)mats, (const u64*)heights, (const u64*)widths, n_mats, 0, true, false);
        memcpy(root32, pd->root, 32);
        *out = pd.release();
    });
}
int msgpu_commit_ldes_dev(msgpu_ctx* h, uint64_t* const* ldes, const uint64_t* heights, const uint64_t* widths,
                          uint64_t n_mats, int take_ownership, msgpu_pdata** out, uint8_t* root32) {
    return msgpu_commit_ldes_blocks_dev(h, ldes, heights, widths, n_mats, 0, nullptr, nullptr, take_ownership, out, root32);
}
// The same where some matrices are still column blocks: block_ptrs[i * n_blocks + b] / block_widths[i * n_blocks + b], b <
// n_blocks, are the dense heights[i] x width_b column blocks of matrix i in column order (all null for a matrix that is already
// in ldes[i]). Such a matrix is WRITTEN to ldes[i] by the pass that hashes its rows (merkle.cu, AsmList): the row shard of a
// column-sharded LDE is assembled from the peers' blocks (pointers from msgpu_peers_ptr) while it is committed.
int msgpu_commit_ldes_blocks_dev(msgpu_ctx* h, uint64_t* const* ldes, const uint64_t* heights, const uint64_t* widths, uint64_t n_mats,
                                 uint64_t n_blocks, const uint64_t* const* block_ptrs, const uint64_t* block_widths, int take_ownership,
                                 msgpu_pdata** out, uint8_t* root32) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(n_mats > 0, "commit_ldes: no matrices given");
        MSG_REQUIRE(n_blocks <= 16 && (n_blocks == 0 || (block_ptrs && block_widths)), "commit_ldes: bad column-block list");
        auto pd = std::make_unique<msgpu_pdata>();
        for (u64 i = 0; i < n_mats; i++) {
            check_shape(heights[i], widths[i]);
            pd->mats.push_back(msgpu_pdata::Mat{(u64*)ldes[i], heights[i], widths[i]});
            if (n_blocks == 0 || !block_ptrs[i * n_blocks]) continue;
            for (u64 b = 0; b < n_blocks; b++) {
                MSG_REQUIRE(block_ptrs[i * n_blocks + b] || block_widths[i * n_blocks + b] == 0, "commit_ldes: null column block");
                pd->mats.back().blocks.push_back({(const u64*)block_ptrs[i * n_blocks + b], block_widths[i * n_blocks + b]});
            }
        }
        // root32 == NULL: stream-ordered, no read-back (the root is the last digest of msgpu_pdata_digests): a row shard's
        // subtree root goes straight into a device all-gather
        if (root32) mmcs_build(c, pd.get());
        else mmcs_build_async(c, pd.get());
        if (take_ownership)
            for (auto& m : pd->mats) m.own = DevBuf(c, (void*)m.ptr);
        if (root32) memcpy(root32, pd->root, 32);
        *out = pd.release();
    });
}

void msgpu_pdata_free(msgpu_pdata* pd) { delete pd; }
uint64_t msgpu_pdata_num_matrices(const msgpu_pdata* pd) { return pd->mats.size(); }
int msgpu_pdata_matrix(const msgpu_pdata* pd, uint64_t idx, uint64_t** dev_ptr, uint64_t* rows, uint64_t* cols) {
    return guard([&] {
        MSG_REQUIRE(idx < pd->mats.size(), "pdata_matrix: index out of range");
        if (dev_ptr) *dev_ptr = (uint64_t*)pd->mats[idx].ptr;
        if (rows) *rows = pd->mats[idx].height;
        if (cols) *cols = pd->mats[idx].width;
    });
}
int msgpu_pdata_read_rows(msgpu_ctx* h, const msgpu_pdata* pd, uint64_t idx, uint64_t row0, uint64_t nrows, uint64_t* out) {
    return guard([&] {
        MSG_REQUIRE(idx < pd->mats.size(), "pdata_read_rows: index out of range");
        auto& m = pd->mats[idx];
        MSG_REQUIRE(row0 <= m.height && nrows <= m.height - row0, "pdata_read_rows: rows out of range");
        if (nrows * m.width == 0) return;
        MSG_CUDA(cudaMemcpyAsync(out, m.ptr + row0 * m.width, nrows * m.width * 8, cudaMemcpyDeviceToHost, h->c.stream));
        h->c.sync();
    });
}
uint64_t msgpu_pdata_num_layers(const msgpu_pdata* pd) { return pd->layer_len.size(); }
uint64_t msgpu_pdata_layer_len(const msgpu_pdata* pd, uint64_t layer) {
    return layer < pd->layer_len.size() ? pd->layer_len[layer] : 0;
}
int msgpu_pdata_read_layer(msgpu_ctx* h, const msgpu_pdata* pd, uint64_t layer, uint8_t* out) {
    return guard([&] {
        MSG_REQUIRE(layer < pd->layer_len.size(), "pdata_read_layer: layer out of range");
        MSG_CUDA(cudaMemcpyAsync(out, pd->digests.bytes() + pd->layer_off[layer] * 32, pd->layer_len[layer] * 32,
                                 cudaMemcpyDeviceToHost, h->c.stream));
        h->c.sync();
    });
}
int msgpu_open_batch(msgpu_ctx* h, const msgpu_pdata* pd, const uint64_t* indices, uint64_t n_idx, uint64_t* opened_out,
                     uint8_t* proof_out) {
    return guard([&] { mmcs_open_batch(h->c, pd, (const u64*)indices, n_idx, (u64*)opened_out, proof_out); });
}

int msgpu_open_batch_multi(msgpu_ctx* h, const msgpu_pdata* const* pds, const uint32_t* shifts, uint64_t n_trees,
                           const uint64_t* indices, uint64_t n_idx, uint64_t* opened_out, uint8_t* proof_out) {
    return guard([&] {
        MSG_REQUIRE(pds && shifts && indices, "open_batch_multi: null argument");
        mmcs_open_multi(h->c, pds, (const u32*)shifts, n_trees, (const u64*)indices, n_idx, (u64*)opened_out, proof_out);
    });
}

int msgpu_blake3_compress_raw(msgpu_ctx* h, const uint32_t* state16, const uint32_t* msg16, uint32_t* out16) {
    return guard([&] {
        Ctx& c = h->c;
        DevBuf buf(c, 48 * 4);
        u32* d = (u32*)buf.p;
        MSG_CUDA(cudaMemcpyAsync(d, state16, 64, cudaMemcpyHostToDevice, c.stream));
        MSG_CUDA(cudaMemcpyAsync(d + 16, msg16, 64, cudaMemcpyHostToDevice, c.stream));
        b3_compress_raw_dev(c, d, d + 16, d + 32);
        MSG_CUDA(cudaMemcpyAsync(out16, d + 32, 64, cudaMemcpyDeviceToHost, c.stream));
        c.sync();
    });
}

}  // extern "C"
