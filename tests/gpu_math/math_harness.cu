// tests/gpu_math/math_harness.cu — batch entry points onto the per-thread field and lattice math of
// kyber-rs_b200/csrc (fe.cuh, sc.cuh, half.cuh).  TEST INFRASTRUCTURE ONLY: never linked into the product library.
//
// tests/test_gpu_field_edges.py builds this one source three ways: as plain host C++ with KB_HOST_EMU (the twin of
// every PTX carry chain), and with nvcc for sm_100a under the two define sets the product's translation units use
// (the default row order, and -DKB_FE_MUL_RIP -DKB_FE_SQ_RIP -DKB_FE_SUBMASK of the verify and key-set units).  Every
// entry takes host arrays, runs one item per thread (per loop iteration on the host) and returns 0 or a CUDA error
// code; it never aborts.  The field ops return the RAW 8-word result, before canonicalisation, so that the device
// bodies can be compared bit for bit with the host build.
#include <stddef.h>
#include <stdint.h>
#include "half.cuh"   // fe.cuh, sc.cuh; found through -I kyber-rs_b200/csrc

// fe_batch ops; reductions take the 512-bit value (b : a)
enum {
    OP_MUL, OP_SQ, OP_ADD, OP_SUB, OP_NEG,
    OP_MUL_ROWS, OP_MUL_RIP, OP_MUL_KARATSUBA, OP_SQ_ROWS, OP_SQ_RIP,
    OP_REDUCE512_MUL, OP_REDUCE512_SHIFT,
    OP_CANON, OP_IS_NEGATIVE, OP_IS_ZERO, OP_INVERT, OP_POW22523,
    FE_NOPS
};
#define HARNESS_EINVAL 1   // cudaErrorInvalidValue

KB_FN void fe_apply(int op, uint32_t* out, const uint32_t* a, const uint32_t* b)
{
    fe x, y, r;
    KB_UNROLL
    for (int i = 0; i < 8; i++) {
        x.v[i] = a[i];
        y.v[i] = b[i];
    }
    switch (op) {
    case OP_MUL: fe_mul(r, x, y); break;
    case OP_SQ: fe_sq(r, x); break;
    case OP_ADD: fe_add(r, x, y); break;
    case OP_SUB: fe_sub(r, x, y); break;
    case OP_NEG: fe_neg(r, x); break;
    case OP_MUL_ROWS: fe_mul_rows(r, x, y); break;
    case OP_MUL_RIP: fe_mul_rip(r, x, y); break;
    case OP_MUL_KARATSUBA: fe_mul_karatsuba(r, x, y); break;
    case OP_SQ_ROWS: fe_sq_rows(r, x); break;
    case OP_SQ_RIP: fe_sq_rip(r, x); break;
    case OP_REDUCE512_MUL:
    case OP_REDUCE512_SHIFT: {
        uint32_t t[16];
        KB_UNROLL
        for (int i = 0; i < 8; i++) {
            t[i] = x.v[i];
            t[8 + i] = y.v[i];
        }
        if (op == OP_REDUCE512_MUL) fe_reduce512_mul(r, t);
        else fe_reduce512_shift(r, t);
        break;
    }
    case OP_CANON: fe_canon(r, x); break;
    case OP_IS_NEGATIVE: fe_set(r, fe_is_negative(x)); break;
    case OP_IS_ZERO: fe_set(r, fe_is_zero(x)); break;
    case OP_INVERT: fe_invert(r, x); break;
    default: fe_pow22523(r, x); break;   // OP_POW22523
    }
    KB_UNROLL
    for (int i = 0; i < 8; i++) out[i] = r.v[i];
}

// sc_half of h[0..8): out[0..8) = u, out[8..16) = |v|, out[16] = vneg, out[17] = bits
#define HALF_OUT_WORDS 18
KB_FN void half_apply(uint32_t* out, const uint32_t* h)
{
    uint32_t hw[8];
    KB_UNROLL
    for (int i = 0; i < 8; i++) hw[i] = h[i];
    kb_halfsc o;
    sc_half(o, hw);
    KB_UNROLL
    for (int i = 0; i < 8; i++) {
        out[i] = o.u[i];
        out[8 + i] = o.v[i];
    }
    out[16] = o.vneg;
    out[17] = (uint32_t)o.bits;
}

#if defined(KB_HOST_EMU)

extern "C" int fe_batch(int op, size_t n, const uint32_t* a, const uint32_t* b, uint32_t* out_raw)
{
    if (op < 0 || op >= FE_NOPS) return HARNESS_EINVAL;
    for (size_t i = 0; i < n; i++) fe_apply(op, out_raw + 8 * i, a + 8 * i, b + 8 * i);
    return 0;
}
extern "C" int half_batch(size_t n, const uint32_t* h, uint32_t* out)
{
    for (size_t i = 0; i < n; i++) half_apply(out + HALF_OUT_WORDS * i, h + 8 * i);
    return 0;
}

#else

#define HARNESS_THREADS 128

static __global__ void k_fe_batch(int op, size_t n, const uint32_t* a, const uint32_t* b, uint32_t* out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) fe_apply(op, out + 8 * i, a + 8 * i, b + 8 * i);
}
static __global__ void k_half_batch(size_t n, const uint32_t* h, uint32_t* out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) half_apply(out + HALF_OUT_WORDS * i, h + 8 * i);
}
static unsigned harness_blocks(size_t n) { return (unsigned)((n + HARNESS_THREADS - 1) / HARNESS_THREADS); }

extern "C" int fe_batch(int op, size_t n, const uint32_t* a, const uint32_t* b, uint32_t* out_raw)
{
    if (op < 0 || op >= FE_NOPS) return HARNESS_EINVAL;
    if (n == 0) return 0;
    const size_t bytes = 32 * n;
    uint32_t *da = nullptr, *db = nullptr, *dout = nullptr;
    cudaError_t e = cudaMalloc(&da, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&db, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&dout, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(da, a, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(db, b, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        k_fe_batch<<<harness_blocks(n), HARNESS_THREADS>>>(op, n, da, db, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(out_raw, dout, bytes, cudaMemcpyDeviceToHost);
    cudaFree(da);
    cudaFree(db);
    cudaFree(dout);
    return (int)e;
}
extern "C" int half_batch(size_t n, const uint32_t* h, uint32_t* out)
{
    if (n == 0) return 0;
    uint32_t *dh = nullptr, *dout = nullptr;
    cudaError_t e = cudaMalloc(&dh, 32 * n);
    if (e == cudaSuccess) e = cudaMalloc(&dout, 4 * HALF_OUT_WORDS * n);
    if (e == cudaSuccess) e = cudaMemcpy(dh, h, 32 * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        k_half_batch<<<harness_blocks(n), HARNESS_THREADS>>>(n, dh, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(out, dout, 4 * HALF_OUT_WORDS * n, cudaMemcpyDeviceToHost);
    cudaFree(dh);
    cudaFree(dout);
    return (int)e;
}

#endif
