// Peer memory over NVLink / NVSwitch: symmetric device windows mapped into every rank of one node with CUDA IPC, so that the
// kernels of the row-sharded prover (host/rowshard_backend.hpp) read their inputs from, and write their results into, the other
// GPUs' HBM directly instead of going through pack -> NCCL all-to-all -> unpack:
//   * k_peer_pack_push turns a rank's natural-order row block into column blocks written straight into the owners' windows,
//   * k_peer_pull_interleave assembles a rank's row shard from the peers' column blocks of the LDE with remote loads,
//     (both sides of the transfer are whole lines: an NTT pass that gathered / scattered its 8-56-byte row segments itself
//     ran at 190 GB/s over NVLink, profiles/rowshard_step_r2.md)
//   * 32-byte subtree roots and other small per-rank results are written into every peer's window (k_peer_put),
//   * ordering is a flag barrier in peer memory (k_peer_barrier): one store per peer, one spin per peer, no host round trip.
// One process per GPU; the 64-byte IPC handles travel once per window over the caller's host all-gather. The allocator inside a
// window is deterministic (first fit, lowest offset): every rank performs the same sequence of calls with the same sizes, so a
// block has the same (segment, offset) on every rank and no addresses are ever exchanged.
#include "capi_common.hpp"
#include "peer_heap.hpp"

#include <cstring>
#include <map>

using namespace msg;

namespace {
constexpr int kMaxPeers = MSGPU_MAX_PEERS;
constexpr size_t kFlagPage = 4096;      // start of segment 0: barrier flags, error word, root ring
constexpr size_t kErrOff = 512;         // u32 error word
constexpr size_t kRingOff = 1024;       // 2 slots x kMaxPeers x 32 bytes

struct PeerBases {
    char* p[kMaxPeers];
};

// Every rank stores `epoch` into slot `rank` of every peer's flag array, then waits until its own array shows `epoch` in every
// slot. Launched behind the work whose writes it publishes: a kernel boundary orders those writes before the flag stores, and
// the consumer's next kernel starts after its spin has seen the flags. A bounded spin (about 4 s) turns a lost peer into an
// error word instead of a hung device.
__global__ void k_peer_barrier(PeerBases b, int rank, int world, unsigned long long epoch) {
    const int e = threadIdx.x;
    if (e >= world) return;
    __threadfence_system();
    volatile unsigned long long* theirs = (volatile unsigned long long*)(b.p[e]) + rank;
    *theirs = epoch;
    __threadfence_system();
    volatile unsigned long long* mine = (volatile unsigned long long*)(b.p[rank]) + e;
    const long long t0 = clock64();
    while (*mine < epoch) {
        if (clock64() - t0 > (8ll << 30)) {
            *(volatile unsigned*)(b.p[rank] + kErrOff) = 1u;
            break;
        }
        __nanosleep(40);
    }
    __threadfence_system();
}

// dst_e[off + rank * words + i] = src[i] on every peer e (an all-gather by remote stores), 8-byte words
__global__ void k_peer_put(PeerBases b, size_t off_bytes, const u64* __restrict__ src, u64 words, int rank, int world) {
    const u64 total = words * (u64)world;
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (u64)gridDim.x * blockDim.x) {
        const int e = (int)(t / words);
        const u64 i = t % words;
        ((u64*)(b.p[e] + off_bytes))[(u64)rank * words + i] = src[i];
    }
}

// out_b[r][c] = in[r][col0_b + c]: the row block is read once, coalesced; consecutive threads write consecutive addresses of one
// destination block except at the block boundaries of a row
struct PushParams {
    const u64* in;
    u64* out[kMaxPeers];
    u32 col0[kMaxPeers + 1];
    u32 n_blocks;
    u64 rows;
};
__global__ void __launch_bounds__(256) k_peer_pack_push(const __grid_constant__ PushParams p) {
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
// out[r][col0_b + c] = blocks[b][r][c]
struct PullParams {
    const u64* blocks[kMaxPeers];
    u32 col0[kMaxPeers + 1];
    u32 n_blocks;
    u64 rows;
    u64* out;
};
__global__ void __launch_bounds__(256) k_peer_pull_interleave(const __grid_constant__ PullParams p) {
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
}  // namespace

struct msgpu_peers {
    Ctx* c = nullptr;
    int rank = 0, world = 1;
    struct Seg {
        size_t bytes = 0;
        char* base[kMaxPeers] = {};
        bool opened = false;
        bool ipc = true;   // the peers' bases are CUDA-IPC mappings (closed at teardown); false: raw pointers of this process
        FirstFitHeap heap;
    };
    std::vector<Seg> segs;
    unsigned long long epoch = 0, ring = 0;
    PeerBases flag_bases() const {
        PeerBases b{};
        for (int e = 0; e < world; e++) b.p[e] = segs[0].base[e];
        return b;
    }
};

namespace msg {
}  // namespace msg

extern "C" {

int msgpu_peers_create(msgpu_ctx* h, int32_t rank, int32_t world, msgpu_peers** out) {
    return guard([&] {
        MSG_REQUIRE(out && world >= 1 && world <= kMaxPeers && rank >= 0 && rank < world, "peers: bad rank / world");
        auto* p = new msgpu_peers();
        p->c = &h->c;
        p->rank = rank;
        p->world = world;
        *out = p;
    });
}

// A new window of `bytes` on this device (collective: every rank creates one of the same size, then exchanges the handles).
int msgpu_peers_segment_create(msgpu_peers* p, uint64_t bytes, uint8_t* handle64) {
    return guard([&] {
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
        MSG_REQUIRE(p && handle64 && bytes >= 2 * kFlagPage, "peers: bad segment size");
        MSG_REQUIRE(p->segs.empty() || p->segs.back().opened, "peers: the previous segment was never opened");
        MSG_CUDA(cudaSetDevice(p->c->device));
        msgpu_peers::Seg s;
        s.bytes = (size_t)bytes;
        void* base = nullptr;
        MSG_CUDA(cudaMalloc(&base, s.bytes));
        s.base[p->rank] = (char*)base;
        size_t first = 0;
        if (p->segs.empty()) {
            MSG_CUDA(cudaMemset(base, 0, kFlagPage));
            first = kFlagPage;
        }
        MSG_CUDA(cudaDeviceSynchronize());
        s.heap = FirstFitHeap(first, s.bytes);
        cudaIpcMemHandle_t hd;
        cudaError_t e = cudaIpcGetMemHandle(&hd, base);
        if (e != cudaSuccess) {
            cudaFree(base);
            throw Error(MSGPU_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
        }
        memcpy(handle64, &hd, 64);
        p->segs.push_back(std::move(s));
    });
}

// handles: world x 64 bytes in rank order (from the host all-gather of what msgpu_peers_segment_create returned)
int msgpu_peers_segment_open(msgpu_peers* p, const uint8_t* handles) {
    return guard([&] {
        MSG_REQUIRE(p && handles && !p->segs.empty() && !p->segs.back().opened, "peers: no segment to open");
        MSG_CUDA(cudaSetDevice(p->c->device));
        auto& s = p->segs.back();
        for (int e = 0; e < p->world; e++) {
            if (e == p->rank) continue;
            cudaIpcMemHandle_t hd;
            memcpy(&hd, handles + 64 * (size_t)e, 64);
            void* ptr = nullptr;
            cudaError_t err = cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess);
            if (err != cudaSuccess) {
                (void)cudaGetLastError();
                throw Error(MSGPU_ERR_CUDA, std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(e) + "): " + cudaGetErrorString(err));
            }
            s.base[e] = (char*)ptr;
        }
        s.opened = true;
    });
}

// The same for ranks that live in ONE process (several contexts / streams, one or several devices with peer access enabled by
// the caller): bases[e] = address of rank e's window, as returned by msgpu_peers_ptr(their peers object, segment, 0, e).
int msgpu_peers_segment_open_local(msgpu_peers* p, void* const* bases) {
    return guard([&] {
        MSG_REQUIRE(p && bases && !p->segs.empty() && !p->segs.back().opened, "peers: no segment to open");
        auto& s = p->segs.back();
        for (int e = 0; e < p->world; e++) {
            if (e == p->rank) continue;
            MSG_REQUIRE(bases[e], "peers: null window address");
            s.base[e] = (char*)bases[e];
        }
        s.ipc = false;
        s.opened = true;
    });
}

uint64_t msgpu_peers_num_segments(const msgpu_peers* p) { return p->segs.size(); }

// Deterministic first fit. Returns 1 (not an error: no last-error text) when no window has room: the caller grows collectively.
int msgpu_peers_alloc(msgpu_peers* p, uint64_t bytes, uint32_t* seg, uint64_t* off) {
    int rc = 1;
    int g = guard([&] {
        MSG_REQUIRE(p && seg && off, "peers: null argument");
        for (size_t s = 0; s < p->segs.size(); s++) {
            auto& sg = p->segs[s];
            if (!sg.opened) continue;
            const size_t o = sg.heap.alloc((size_t)bytes);
            if (o == FirstFitHeap::npos) continue;
            *seg = (uint32_t)s;
            *off = o;
            rc = 0;
            return;
        }
    });
    return g != MSGPU_OK ? g : rc;
}

int msgpu_peers_free_block(msgpu_peers* p, uint32_t seg, uint64_t off) {
    return guard([&] {
        MSG_REQUIRE(p && seg < p->segs.size(), "peers: no such segment");
        MSG_REQUIRE(p->segs[seg].heap.free((size_t)off), "peers: not a live block");
    });
}

// address of (segment, offset) in rank `peer`'s window as mapped HERE (peer == own rank: the local address)
void* msgpu_peers_ptr(const msgpu_peers* p, uint32_t seg, uint64_t off, int32_t peer) {
    if (!p || seg >= p->segs.size() || peer < 0 || peer >= p->world || off >= p->segs[seg].bytes) return nullptr;
    return p->segs[seg].base[peer] + off;
}

int msgpu_peers_barrier(msgpu_peers* p) {
    return guard([&] {
        MSG_REQUIRE(p && !p->segs.empty() && p->segs[0].opened, "peers: no window");
        Ctx& c = *p->c;
        p->epoch++;
        StageScope ss(c, "exchange");
        launch(c, "k_peer_barrier", k_peer_barrier, 1, 32, 0, p->flag_bases(), p->rank, p->world, p->epoch);
    });
}

// All-gather by remote stores: every peer's block (seg, off) receives `bytes` (a multiple of 8) from this rank at
// off + rank * bytes. Not ordered against the peers: follow with msgpu_peers_barrier.
int msgpu_peers_put(msgpu_peers* p, const void* src_dev, uint32_t seg, uint64_t off, uint64_t bytes) {
    return guard([&] {
        MSG_REQUIRE(p && src_dev && seg < p->segs.size() && p->segs[seg].opened && bytes % 8 == 0, "peers: bad put");
        MSG_REQUIRE(off + bytes * (uint64_t)p->world <= p->segs[seg].bytes, "peers: put outside the segment");
        if (bytes == 0) return;
        Ctx& c = *p->c;
        PeerBases b{};
        for (int e = 0; e < p->world; e++) b.p[e] = p->segs[seg].base[e];
        const u64 words = bytes / 8, total = words * (u64)p->world;
        StageScope ss(c, "exchange");
        launch(c, "k_peer_put", k_peer_put, (unsigned)std::min<u64>((total + 255) / 256, (u64)c.sm_count * 8), 256, 0, b, (size_t)off,
               (const u64*)src_dev, words, p->rank, p->world);
    });
}

// The 32-byte subtree roots of a row-sharded commitment: this rank's root goes into slot `rank` of the current ring entry on
// every peer; returns the local address of the entry (world x 32 bytes, complete after the next msgpu_peers_barrier). Two ring
// entries: a peer can run at most one commitment ahead of the slowest rank (it needs that rank's barrier flag to go further).
int msgpu_peers_put_root(msgpu_peers* p, const uint8_t* root_dev, uint8_t** gathered_dev) {
    return guard([&] {
        MSG_REQUIRE(p && root_dev && gathered_dev && !p->segs.empty() && p->segs[0].opened, "peers: no window");
        Ctx& c = *p->c;
        const size_t off = kRingOff + (size_t)(p->ring++ & 1u) * kMaxPeers * 32;
        StageScope ss(c, "exchange");
        launch(c, "k_peer_put", k_peer_put, 1, 64, 0, p->flag_bases(), off, (const u64*)root_dev, 4, p->rank, p->world);
        *gathered_dev = (uint8_t*)(p->segs[0].base[p->rank] + off);
    });
}

// 0 = every barrier so far completed; MSGPU_ERR_CUDA = a peer never arrived (call after a stream synchronisation)
int msgpu_peers_check(msgpu_peers* p) {
    return guard([&] {
        MSG_REQUIRE(p && !p->segs.empty(), "peers: no window");
        unsigned err = 0;
        MSG_CUDA(cudaMemcpyAsync(&err, p->segs[0].base[p->rank] + kErrOff, 4, cudaMemcpyDeviceToHost, p->c->stream));
        MSG_CUDA(cudaStreamSynchronize(p->c->stream));
        if (err) throw Error(MSGPU_ERR_CUDA, "peers: a barrier timed out (a peer never arrived)");
    });
}

// Row blocks -> column blocks by remote stores. src: this rank's natural-order row block (rows x width, local). Block (seg, off)
// of rank e's window is e's dense COLUMN block (rows * world x wd_e, wd_e = e's share of the columns: the first width % world
// ranks hold one more); this rank writes its rows [rank * rows, (rank + 1) * rows) of every peer's block -- contiguous in the
// destination, so the NVLink stores are full lines. Follow with msgpu_peers_barrier.
int msgpu_peers_pack_push(msgpu_peers* p, const uint64_t* src_dev, uint64_t rows, uint64_t width, uint32_t seg, uint64_t off) {
    return guard([&] {
        MSG_REQUIRE(p && src_dev && seg < p->segs.size() && p->segs[seg].opened && width >= 1, "peers: bad pack_push");
        if (rows == 0) return;
        Ctx& c = *p->c;
        const u64 N = (u64)p->world, base = width / N, rem = width % N;
        PushParams pp{};
        pp.in = (const u64*)src_dev;
        pp.rows = rows;
        pp.n_blocks = (u32)N;
        u64 col = 0;
        for (u64 e = 0; e < N; e++) {
            const u64 wd = base + (e < rem ? 1 : 0);
            MSG_REQUIRE(off + rows * N * wd * 8 <= p->segs[seg].bytes, "peers: pack_push outside the segment");
            pp.col0[e] = (u32)col;
            pp.out[e] = (u64*)(p->segs[seg].base[e] + off) + (u64)p->rank * rows * wd;
            col += wd;
        }
        pp.col0[N] = (u32)width;
        StageScope ss(c, "exchange");
        launch(c, "k_peer_pack_push", k_peer_pack_push, (unsigned)std::min<u64>((rows * width + 255) / 256, (u64)c.sm_count * 16), 256, 0, pp);
    });
}

// Column blocks -> row shard by remote loads. Block (seg, off) of rank e's window is e's dense column block of the LDE
// (rows * world x wd_e); this rank reads rows [rank * rows, (rank + 1) * rows) of every peer's block (contiguous: full-line NVLink
// loads) and writes its shard dst (rows x width, local, row-major over all columns). Needs a barrier before (the peers' LDEs are
// complete) and one after, before the peers release their blocks.
int msgpu_peers_pull_interleave(msgpu_peers* p, uint32_t seg, uint64_t off, uint64_t rows, uint64_t width, uint64_t* dst_dev) {
    return guard([&] {
        MSG_REQUIRE(p && dst_dev && seg < p->segs.size() && p->segs[seg].opened && width >= 1, "peers: bad pull_interleave");
        if (rows == 0) return;
        Ctx& c = *p->c;
        const u64 N = (u64)p->world, base = width / N, rem = width % N;
        PullParams pp{};
        pp.out = (u64*)dst_dev;
        pp.rows = rows;
        pp.n_blocks = (u32)N;
        u64 col = 0;
        for (u64 e = 0; e < N; e++) {
            const u64 wd = base + (e < rem ? 1 : 0);
            MSG_REQUIRE(off + rows * N * wd * 8 <= p->segs[seg].bytes, "peers: pull_interleave outside the segment");
            pp.col0[e] = (u32)col;
            pp.blocks[e] = (const u64*)(p->segs[seg].base[e] + off) + (u64)p->rank * rows * wd;
            col += wd;
        }
        pp.col0[N] = (u32)width;
        StageScope ss(c, "exchange");
        launch(c, "k_peer_pull_interleave", k_peer_pull_interleave, (unsigned)std::min<u64>((rows * width + 255) / 256, (u64)c.sm_count * 16), 256,
               0, pp);
    });
}

// Teardown is local: the peers' mappings are closed, then this rank's windows are freed. Every rank has passed a barrier behind
// its last access to any window by then (a commitment ends with one), so no transfer is in flight. The CUDA documentation asks
// importers to close before the exporter frees; that order is NOT enforced across ranks here (it would take a host collective
// inside a destructor, which hangs when a rank has already failed). No access follows the free on any rank, and every run on
// driver 580 (tests/test_gpu_peer.py, bench.py at N = 2, 4, 8: several provers created and destroyed per process) is clean.
void msgpu_peers_destroy(msgpu_peers* p) {
    if (!p) return;
    cudaSetDevice(p->c->device);
    cudaStreamSynchronize(p->c->stream);
    for (auto& s : p->segs) {
        for (int e = 0; e < p->world; e++) {
            if (!s.base[e]) continue;
            if (e == p->rank) cudaFree(s.base[e]);
            else if (s.ipc) cudaIpcCloseMemHandle(s.base[e]);
        }
    }
    delete p;
}

}  // extern "C"
