// Integer-pipe peak microbenchmarks (measurement support, not on the proving path). The NTT and BLAKE3 kernels are bound
// by the INT32 pipes, for which MEASURED_PEAKS.json has no entry; msgpu_measure_int_peak times three dependency-free
// instruction streams with CUDA events so that bench.py can report an integer roofline next to the HBM one:
//   [0] ALU pipe only   : LOP3 + SHF   (xor / funnel-shift, cannot issue on the FMA pipe)
//   [1] FMA pipe only   : IMAD         (32-bit multiply-add)
//   [2] both, 1 : 1     : the best case for integer code, one instruction per scheduler per clock
// Results are in G thread-instructions per second for the whole GPU.
#include "capi_common.hpp"

namespace msg {

constexpr int kPeakIters = 4096;
constexpr int kPeakIlp = 8;

template <int MODE>
__global__ void __launch_bounds__(256) k_int_peak(u32* out, u32 seed) {
    u32 x[kPeakIlp], y[kPeakIlp];
#pragma unroll
    for (int i = 0; i < kPeakIlp; i++) { x[i] = seed + threadIdx.x * 31u + i; y[i] = seed * 7u + blockIdx.x + i * 3u; }
    for (int it = 0; it < kPeakIters; it++) {
#pragma unroll
        for (int i = 0; i < kPeakIlp; i++) {
            if (MODE == 0 || MODE == 2) {
                asm volatile("xor.b32 %0, %0, %1;" : "+r"(x[i]) : "r"(y[i]));
                asm volatile("shf.l.wrap.b32 %0, %0, %0, 7;" : "+r"(x[i]));
            }
            if (MODE == 1 || MODE == 2) {
                asm volatile("mad.lo.u32 %0, %0, %1, %1;" : "+r"(y[i]) : "r"(x[i]));
                asm volatile("mad.lo.u32 %0, %0, %1, %0;" : "+r"(y[i]) : "r"(x[i]));
            }
        }
    }
    u32 acc = 0;
#pragma unroll
    for (int i = 0; i < kPeakIlp; i++) acc ^= x[i] + y[i];
    if (acc == 0x12345678u) out[0] = acc;  // keeps the streams alive
}

template <int MODE>
static double run_peak(Ctx& c, u32* d_out) {
    const unsigned blocks = (unsigned)c.sm_count * 8;
    const double per_thread = (double)kPeakIters * kPeakIlp * (MODE == 2 ? 4.0 : 2.0);
    cudaEvent_t a, b;
    MSG_CUDA(cudaEventCreate(&a));
    MSG_CUDA(cudaEventCreate(&b));
    launch(c, "k_int_peak", k_int_peak<MODE>, blocks, 256, 0, d_out, 1u);  // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        MSG_CUDA(cudaEventRecord(a, c.stream));
        launch(c, "k_int_peak", k_int_peak<MODE>, blocks, 256, 0, d_out, 2u + rep);
        MSG_CUDA(cudaEventRecord(b, c.stream));
        MSG_CUDA(cudaEventSynchronize(b));
        float ms = 0;
        MSG_CUDA(cudaEventElapsedTime(&ms, a, b));
        best = std::min(best, ms);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    return per_thread * blocks * 256.0 / (best * 1e-3) / 1e9;
}

}  // namespace msg

using namespace msg;

extern "C" int msgpu_measure_int_peak(msgpu_ctx* h, double* out3) {
    return guard([&] {
        Ctx& c = h->c;
        MSG_REQUIRE(out3 != nullptr, "measure_int_peak: null output");
        DevBuf buf(c, 64);
        out3[0] = run_peak<0>(c, (u32*)buf.p);
        out3[1] = run_peak<1>(c, (u32*)buf.p);
        out3[2] = run_peak<2>(c, (u32*)buf.p);
    });
}
