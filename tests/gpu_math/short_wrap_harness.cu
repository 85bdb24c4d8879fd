// tests/gpu_math/short_wrap_harness.cu — batch entry point onto the short-wrap field bodies of kyber-rs_b200/csrc/fe.cuh
// (fe_sw) and the exact bodies they stand in for.  TEST INFRASTRUCTURE ONLY: never linked into the product library.
//
// tests/test_verify_short_wrap.py builds it like math_harness.cu: as plain host C++ with KB_HOST_EMU, and with nvcc for
// sm_100a under the default bodies and under -DKB_FE_MUL_RIP -DKB_FE_SQ_RIP -DKB_FE_SUBMASK (the verify unit's).  One
// item per thread; returns 0 or a CUDA error code and never aborts.  Results are RAW words, before canonicalisation.
#include <stddef.h>
#include <stdint.h>
#include "fe.cuh"   // found through -I kyber-rs_b200/csrc

// ops: 0 mul, 1 sq, 2 add, 3 sub, 4 dbl, 5 neg, 6 reduction of the 512-bit value (b : a)
#define SW_NOPS 7
#define HARNESS_EINVAL 1   // cudaErrorInvalidValue

template <class F>
KB_FN void sw_run(int op, fe& r, const fe& x, const fe& y, F& fo)
{
    switch (op) {
    case 0: fe_mul(r, x, y, fo); break;
    case 1: fe_sq(r, x, fo); break;
    case 2: fe_add(r, x, y, fo); break;
    case 3: fe_sub(r, x, y, fo); break;
    case 4: fe_dbl(r, x, fo); break;
    default: fe_neg(r, x, fo); break;
    }
}
// exact = 1: the exact body (ovf = 0), 0: the short-wrap body and its counter
KB_FN void sw_apply(int op, int exact, uint32_t* out, uint32_t* ovf, const uint32_t* a, const uint32_t* b)
{
    fe x, y, r;
    KB_UNROLL
    for (int i = 0; i < 8; i++) {
        x.v[i] = a[i];
        y.v[i] = b[i];
    }
    fe_sw sw = {0};
    if (op == 6) {
        uint32_t t[16];
        KB_UNROLL
        for (int i = 0; i < 8; i++) {
            t[i] = x.v[i];
            t[8 + i] = y.v[i];
        }
        if (exact) fe_reduce512_mul(r, t);
        else fe_reduce512_sw(r, t, sw.ovf);
    } else if (exact) {
        fe_ex ex;
        sw_run(op, r, x, y, ex);
    } else {
        sw_run(op, r, x, y, sw);
    }
    KB_UNROLL
    for (int i = 0; i < 8; i++) out[i] = r.v[i];
    *ovf = sw.ovf;
}

#if defined(KB_HOST_EMU)

extern "C" int fe_sw_batch(int op, int exact, size_t n, const uint32_t* a, const uint32_t* b, uint32_t* out_raw, uint32_t* ovf)
{
    if (op < 0 || op >= SW_NOPS) return HARNESS_EINVAL;
    for (size_t i = 0; i < n; i++) sw_apply(op, exact, out_raw + 8 * i, ovf + i, a + 8 * i, b + 8 * i);
    return 0;
}

#else

#define HARNESS_THREADS 128

static __global__ void k_fe_sw_batch(int op, int exact, size_t n, const uint32_t* a, const uint32_t* b, uint32_t* out, uint32_t* ovf)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sw_apply(op, exact, out + 8 * i, ovf + i, a + 8 * i, b + 8 * i);
}

extern "C" int fe_sw_batch(int op, int exact, size_t n, const uint32_t* a, const uint32_t* b, uint32_t* out_raw, uint32_t* ovf)
{
    if (op < 0 || op >= SW_NOPS) return HARNESS_EINVAL;
    if (n == 0) return 0;
    const size_t bytes = 32 * n;
    uint32_t *da = nullptr, *db = nullptr, *dout = nullptr, *dovf = nullptr;
    cudaError_t e = cudaMalloc(&da, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&db, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&dout, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&dovf, 4 * n);
    if (e == cudaSuccess) e = cudaMemcpy(da, a, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(db, b, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        k_fe_sw_batch<<<(unsigned)((n + HARNESS_THREADS - 1) / HARNESS_THREADS), HARNESS_THREADS>>>(op, exact, n, da, db, dout, dovf);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(out_raw, dout, bytes, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(ovf, dovf, 4 * n, cudaMemcpyDeviceToHost);
    cudaFree(da);
    cudaFree(db);
    cudaFree(dout);
    cudaFree(dovf);
    return (int)e;
}

#endif
