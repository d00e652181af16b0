// Test-only device harness for the Goldilocks primitives of multi_stark_b200/csrc/gl.cuh (not part of libmsgpu).
//
// One small kernel per primitive family, dispatched by an op id; gf::mul_pow2 is instantiated for every e in 1..95 because
// its exponent must be a compile-time constant. The extern "C" launchers take host arrays, copy them to the device, run one
// kernel and copy the results back. tests/test_gpu_field.py compiles this file with the library's nvcc flags and compares
// every result with Python ints.
#include <array>
#include <utility>

#include "../multi_stark_b200/csrc/gl.cuh"

using namespace gl;

enum Op : int {
    OP_CANON, OP_ADD_LAZY, OP_SUB_LAZY, OP_ADD, OP_SUB, OP_NEG, OP_REDUCE128_LAZY, OP_MUL, OP_MUL_LAZY, OP_SQR, OP_POW, OP_INV,
    OP_HALVE, OP_GF_ADD, OP_GF_SUB, OP_GF_REDUCE128, OP_GF_MUL, OP_MUL7, OP_POW2_MOD_P, OP_REV_BITS,
    OP_E2_ADD, OP_E2_SUB, OP_E2_MUL, OP_E2_MUL_BASE, OP_E2_INV,
};

__global__ void k_base(int op, const u64* a, const u64* b, u64* out, u64 n) {
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u64 x = a[i], y = b[i];
        u64 r;
        switch (op) {
            case OP_CANON: r = canon(x); break;
            case OP_ADD_LAZY: r = add_lazy(x, y); break;
            case OP_SUB_LAZY: r = sub_lazy(x, y); break;
            case OP_ADD: r = add(x, y); break;
            case OP_SUB: r = sub(x, y); break;
            case OP_NEG: r = neg(x); break;
            case OP_REDUCE128_LAZY: r = reduce128_lazy(x, y); break;  // lo = a, hi = b
            case OP_MUL: r = mul(x, y); break;
            case OP_MUL_LAZY: r = mul_lazy(x, y); break;
            case OP_SQR: r = sqr(x); break;
            case OP_POW: r = pow(x, y); break;
            case OP_INV: r = inv(x); break;
            case OP_HALVE: r = halve(x); break;
            case OP_GF_ADD: r = gf::add(x, y); break;
            case OP_GF_SUB: r = gf::sub(x, y); break;
            case OP_GF_REDUCE128: r = gf::reduce128(x, y); break;
            case OP_GF_MUL: r = gf::mul(x, y); break;
            case OP_MUL7: r = mul7(x); break;
            case OP_POW2_MOD_P: r = gf::pow2_mod_p((int)x); break;
            case OP_REV_BITS: r = rev_bits((u32)x, (u32)y); break;
            default: r = 0xdeadull; break;
        }
        out[i] = r;
    }
}

// extension-field ops: a, b, out hold (c0, c1) pairs; OP_E2_MUL_BASE multiplies by b[2i]
__global__ void k_e2(int op, const u64* a, const u64* b, u64* out, u64 n) {
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const e2 x = e2_make(a[2 * i], a[2 * i + 1]), y = e2_make(b[2 * i], b[2 * i + 1]);
        e2 r;
        switch (op) {
            case OP_E2_ADD: r = e2_add(x, y); break;
            case OP_E2_SUB: r = e2_sub(x, y); break;
            case OP_E2_MUL: r = e2_mul(x, y); break;
            case OP_E2_MUL_BASE: r = e2_mul_base(x, y.a); break;
            case OP_E2_INV: r = e2_inv(x); break;
            default: r = e2_make(0xdeadull, 0xdeadull); break;
        }
        out[2 * i] = r.a;
        out[2 * i + 1] = r.b;
    }
}

template <int E>
__global__ void k_mul_pow2(const u64* x, u64* out, u64 n) {
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        out[i] = gf::mul_pow2(x[i], E);
}
using MulPow2Kernel = void (*)(const u64*, u64*, u64);
template <int... E>
constexpr std::array<MulPow2Kernel, sizeof...(E)> mul_pow2_kernels(std::integer_sequence<int, E...>) {
    return {&k_mul_pow2<E + 1>...};
}
static const std::array<MulPow2Kernel, 95> kMulPow2 = mul_pow2_kernels(std::make_integer_sequence<int, 95>{});

// one acc_mac per lane on the limb state st[5i .. 5i+5), then acc_reduce
__global__ void k_acc_mac(const u32* st, const u64* a, const u64* b, u32* out_st, u64* out, u64 n) {
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        Acc160 s;
        s.l0 = st[5 * i]; s.l1 = st[5 * i + 1]; s.l2 = st[5 * i + 2]; s.l3 = st[5 * i + 3]; s.l4 = st[5 * i + 4];
        const u64 r0 = acc_reduce(s);
        acc_mac(s, a[i], b[i]);
        out_st[5 * i] = s.l0; out_st[5 * i + 1] = s.l1; out_st[5 * i + 2] = s.l2; out_st[5 * i + 3] = s.l3;
        out_st[5 * i + 4] = s.l4;
        out[2 * i] = r0;  // acc_reduce of the state before and after the term
        out[2 * i + 1] = acc_reduce(s);
    }
}

// one thread: `terms` terms of a * b from zero
__global__ void k_acc_repeat(u64 a, u64 b, u64 terms, u32* out_st, u64* out) {
    Acc160 s = acc_zero();
    for (u64 t = 0; t < terms; t++) acc_mac(s, a, b);
    out_st[0] = s.l0; out_st[1] = s.l1; out_st[2] = s.l2; out_st[3] = s.l3; out_st[4] = s.l4;
    out[0] = acc_reduce(s);
}

__global__ void k_pow_lookup(const u64* lo, const u64* hi, u32 h1, const u64* e, u64* out, u64 n) {
    const PowTable t{lo, hi, h1};
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) out[i] = pow_lookup(t, e[i]);
}

namespace {
struct Dev {  // one device copy of a host array; freed on scope exit
    void* p = nullptr;
    size_t bytes;
    cudaError_t err;
    Dev(const void* host, size_t n) : bytes(n) {
        err = cudaMalloc(&p, n ? n : 1);
        if (err == cudaSuccess && host && n) err = cudaMemcpy(p, host, n, cudaMemcpyHostToDevice);
    }
    ~Dev() { cudaFree(p); }
    template <class T> T* as() { return (T*)p; }
};
unsigned grid(u64 n) { return (unsigned)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096) + (n == 0); }

// the first error among the copies, the launch and the kernel's run
int finish(std::initializer_list<const Dev*> bufs) {
    for (const Dev* d : bufs)
        if (d->err != cudaSuccess) return (int)d->err;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    return (int)e;
}
int copy_out(void* host, const Dev& d) {
    cudaError_t e = cudaMemcpyAsync(host, d.p, d.bytes, cudaMemcpyDeviceToHost, 0);
    return (int)(e != cudaSuccess ? e : cudaStreamSynchronize(0));
}
}  // namespace

extern "C" {

int gh_base(int op, const u64* a, const u64* b, u64* out, u64 n) {
    Dev da(a, n * 8), db(b, n * 8), dout(nullptr, n * 8);
    k_base<<<grid(n), 256>>>(op, da.as<u64>(), db.as<u64>(), dout.as<u64>(), n);
    if (int e = finish({&da, &db, &dout})) return e;
    return copy_out(out, dout);
}

int gh_e2(int op, const u64* a, const u64* b, u64* out, u64 n) {
    Dev da(a, n * 16), db(b, n * 16), dout(nullptr, n * 16);
    k_e2<<<grid(n), 256>>>(op, da.as<u64>(), db.as<u64>(), dout.as<u64>(), n);
    if (int e = finish({&da, &db, &dout})) return e;
    return copy_out(out, dout);
}

// e in 1..95
int gh_mul_pow2(int e, const u64* x, u64* out, u64 n) {
    if (e < 1 || e > 95) return -1;
    Dev dx(x, n * 8), dout(nullptr, n * 8);
    kMulPow2[e - 1]<<<grid(n), 256>>>(dx.as<u64>(), dout.as<u64>(), n);
    if (int r = finish({&dx, &dout})) return r;
    return copy_out(out, dout);
}

int gh_acc_mac(const u32* st, const u64* a, const u64* b, u32* out_st, u64* out, u64 n) {
    Dev dst(st, n * 20), da(a, n * 8), db(b, n * 8), dout_st(nullptr, n * 20), dout(nullptr, n * 16);
    k_acc_mac<<<grid(n), 256>>>(dst.as<u32>(), da.as<u64>(), db.as<u64>(), dout_st.as<u32>(), dout.as<u64>(), n);
    if (int e = finish({&dst, &da, &db, &dout_st, &dout})) return e;
    if (int e = copy_out(out_st, dout_st)) return e;
    return copy_out(out, dout);
}

int gh_acc_repeat(u64 a, u64 b, u64 terms, u32* out_st, u64* out) {
    Dev dout_st(nullptr, 20), dout(nullptr, 8);
    k_acc_repeat<<<1, 1>>>(a, b, terms, dout_st.as<u32>(), dout.as<u64>());
    if (int e = finish({&dout_st, &dout})) return e;
    if (int e = copy_out(out_st, dout_st)) return e;
    return copy_out(out, dout);
}

int gh_pow_lookup(const u64* lo, u64 n_lo, const u64* hi, u64 n_hi, u32 h1, const u64* e, u64* out, u64 n) {
    Dev dlo(lo, n_lo * 8), dhi(hi, n_hi * 8), de(e, n * 8), dout(nullptr, n * 8);
    k_pow_lookup<<<grid(n), 256>>>(dlo.as<u64>(), dhi.as<u64>(), h1, de.as<u64>(), dout.as<u64>(), n);
    if (int r = finish({&dlo, &dhi, &de, &dout})) return r;
    return copy_out(out, dout);
}

}  // extern "C"
