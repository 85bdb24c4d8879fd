// capi_signer.cu — signer sets: schnorr::sign / EdDSA::sign under registered secret keys (include/kyber_b200.h)
#define KB_K_SIGNER
// the field-arithmetic bodies of the other signing kernels (capi_verify.cu)
#define KB_FE_MUL_RIP
#define KB_FE_SQ_RIP
#define KB_FE_SUBMASK
#include "ctx.cuh"
#include "kernels.cuh"

// One allocation per signer set: sec[32 nkeys] (x or a), then pk[32 nkeys] (A), then for EdDSA prefix[32 nkeys].  It is
// not part of the context's scratch, so kb_ctx_wipe leaves it alone; kb_signerset_destroy zeroes it.
struct kb_signerset {
    kb_ctx* ctx;
    size_t nkeys;
    int kind;
    size_t bytes;
    uint8_t* mem;
    uint8_t* sec;
    uint8_t* pk;
    uint8_t* prefix;
};

// scratch slot of the EdDSA nonces r between the two kernels of a device call; zeroed on the call's stream at its end
#define KB_SLOT_SIGNER_R 9

// k_signer_stage1, k_compress_batch of R, k_signer_finish on device buffers; the caller has checked the nonce / kind pairing
static int kb_signer_launch(kb_signerset* ss, size_t n, const uint32_t* d_idx, const uint8_t* d_nonces, const uint8_t* d_msg, const uint64_t* d_off, uint8_t* d_sig, uint8_t* d_st,
                            uint32_t* xyz, uint8_t* d_r, uint8_t* d_renc, cudaStream_t st)
{
    kb_ctx* ctx = ss->ctx;
    const unsigned g = kb_blocks(n, KB_THREADS);
    const size_t smem = 64 * 8 * 96;
    if (ss->kind == KB_SIGNER_EDDSA)
        k_signer_stage1<true><<<g, KB_THREADS, smem, st>>>(n, d_idx, ss->nkeys, ss->prefix, nullptr, d_msg, d_off, xyz, d_r, d_st, ctx->base_table);
    else
        k_signer_stage1<false><<<g, KB_THREADS, smem, st>>>(n, d_idx, ss->nkeys, nullptr, d_nonces, d_msg, d_off, xyz, nullptr, d_st, ctx->base_table);
    KB_LAUNCHED();
    k_compress_batch<<<kb_blocks((n + KB_INV_K - 1) / KB_INV_K, KB_THREADS), KB_THREADS, 0, st>>>(n, xyz, d_st, d_renc);
    KB_LAUNCHED();
    k_signer_finish<<<g, KB_THREADS, 0, st>>>(n, d_idx, ss->nkeys, ss->sec, ss->pk, d_renc, d_msg, d_off, ss->kind == KB_SIGNER_EDDSA ? d_r : d_nonces, d_sig);
    KB_LAUNCHED();
    return KB_OK;
}

extern "C" {
int kb_signerset_create(kb_ctx* ctx, size_t nkeys, const uint8_t* keys, int kind, uint8_t* pk_out, kb_signerset** out)
{
    KB_ENTER();
    if (!out) return KB_ERR_ARG;
    *out = nullptr;
    if (nkeys == 0 || !keys || (kind != KB_SIGNER_SCHNORR && kind != KB_SIGNER_EDDSA)) return KB_ERR_ARG;
    const size_t per_key = kind == KB_SIGNER_EDDSA ? 96 : 64;
    if (nkeys > (SIZE_MAX - 256) / per_key) return KB_ERR_NOMEM;
    kb_signerset* ss = (kb_signerset*)calloc(1, sizeof(kb_signerset));
    if (!ss) return KB_ERR_NOMEM;
    ss->ctx = ctx;
    ss->nkeys = nkeys;
    ss->kind = kind;
    ss->bytes = nkeys * per_key;
    const cudaError_t e = cudaMalloc(&ss->mem, ss->bytes);
    if (e != cudaSuccess) {
        kb_fail(ctx, e, "kb_signerset_create: cudaMalloc of the keys");
        free(ss);
        return KB_ERR_NOMEM;
    }
    ss->sec = ss->mem;
    ss->pk = ss->mem + 32 * nkeys;
    ss->prefix = kind == KB_SIGNER_EDDSA ? ss->mem + 64 * nkeys : nullptr;
    // Schnorr: the keys are x itself.  EdDSA: the seeds pass through the pk slots, which the multiplication below overwrites
    // with A, so that no seed is left in device memory.
    uint8_t* stage = kind == KB_SIGNER_EDDSA ? ss->pk : ss->sec;
    int rc = KB_OK;
    cudaError_t ce = cudaMemcpyAsync(stage, keys, 32 * nkeys, cudaMemcpyHostToDevice, ctx->stream);
    if (ce != cudaSuccess) rc = kb_fail(ctx, ce, "kb_signerset_create: copy of the keys");
    if (rc == KB_OK && kind == KB_SIGNER_EDDSA) {
        k_signer_derive<<<kb_blocks(nkeys, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(nkeys, ss->pk, ss->sec, ss->prefix);
        ctx->launches++;
        ce = cudaGetLastError();
        if (ce != cudaSuccess) rc = kb_fail(ctx, ce, "kb_signerset_create: k_signer_derive");
    }
    // A = sec * B by the constant-time fixed-base multiplication (the bytes kb_point_mul_base_batch returns)
    if (rc == KB_OK) rc = kb_dev_point_mul_base(ctx, nkeys, ss->sec, ss->pk, 0, ctx->stream);
    if (rc == KB_OK && pk_out) {
        ce = cudaMemcpyAsync(pk_out, ss->pk, 32 * nkeys, cudaMemcpyDeviceToHost, ctx->stream);
        if (ce != cudaSuccess) rc = kb_fail(ctx, ce, "kb_signerset_create: copy of the public keys");
    }
    if (rc == KB_OK) {
        ce = cudaStreamSynchronize(ctx->stream);
        if (ce != cudaSuccess) rc = kb_fail(ctx, ce, "kb_signerset_create");
    }
    if (rc != KB_OK) {
        kb_signerset_destroy(ss);
        return rc;
    }
    *out = ss;
    return KB_OK;
}
void kb_signerset_destroy(kb_signerset* ss)
{
    if (!ss) return;
    cudaSetDevice(ss->ctx->device);
    cudaDeviceSynchronize();   // sign calls on any stream may still read the keys
    if (ss->mem) {
        // the secret keys do not outlive the set: the zeroing has finished before the memory is released
        if (cudaMemsetAsync(ss->mem, 0, ss->bytes, ss->ctx->stream) == cudaSuccess) cudaStreamSynchronize(ss->ctx->stream);
        cudaFree(ss->mem);
    }
    free(ss);
}
int kb_dev_signerset_sign(kb_signerset* ss, size_t n, const void* d_key_idx, const void* d_nonces, const void* d_msg, const void* d_msg_off, void* d_sig, void* d_status, void* stream)
{
    if (!ss) return KB_ERR_ARG;
    kb_ctx* ctx = ss->ctx;
    if ((ss->kind == KB_SIGNER_SCHNORR) != (d_nonces != nullptr)) return KB_ERR_ARG;
    if (n && (!d_key_idx || !d_msg_off || !d_sig)) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    uint32_t* xyz;
    uint8_t *d_r = nullptr, *d_renc, *d_st = (uint8_t*)d_status;
    KB_SCRATCH(KB_SLOT_XYZ, 96 * n, xyz);
    KB_SCRATCH(8, 32 * n, d_renc);
    if (!d_st) KB_SCRATCH(KB_SLOT_FLAGS, n, d_st);
    if (ss->kind == KB_SIGNER_EDDSA) KB_SCRATCH(KB_SLOT_SIGNER_R, 32 * n, d_r);
    int rc = kb_signer_launch(ss, n, (const uint32_t*)d_key_idx, (const uint8_t*)d_nonces, (const uint8_t*)d_msg, (const uint64_t*)d_msg_off, (uint8_t*)d_sig, d_st, xyz, d_r, d_renc, st);
    // the EdDSA nonces do not outlive the call in scratch, on the error paths either
    if (d_r) {
        const cudaError_t e = cudaMemsetAsync(d_r, 0, 32 * n, st);
        if (rc == KB_OK && e != cudaSuccess) rc = kb_fail(ctx, e, "kb_dev_signerset_sign: zeroing of the nonces");
    }
    KB_DEV_RETURN(st, rc);
}
// staging of kb_signerset_sign_batch; the caller wipes the nonce scratch whatever this returns
static int kb_signer_host_run(kb_signerset* ss, size_t n, const uint32_t* key_idx, const uint8_t* nonces, const uint8_t* msg, const uint64_t* msg_off, size_t mbytes, uint8_t* sig, uint8_t* d_k)
{
    kb_ctx* ctx = ss->ctx;
    uint32_t* d_idx;
    uint8_t *d_m, *d_sig;
    uint64_t* d_off;
    KB_SCRATCH(0, 4 * n, d_idx);
    KB_SCRATCH(1, 64 * n, d_sig);
    KB_SCRATCH(2, mbytes, d_m);
    KB_SCRATCH(3, 8 * (n + 1), d_off);
    if (d_k) KB_H2D(d_k, nonces, 32 * n);
    KB_H2D(d_idx, key_idx, 4 * n);
    if (mbytes) KB_H2D(d_m, msg, mbytes);
    KB_H2D(d_off, msg_off, 8 * (n + 1));
    const int rc = kb_dev_signerset_sign(ss, n, d_idx, d_k, d_m, d_off, d_sig, nullptr, ctx->stream);
    if (rc != KB_OK) return rc;
    KB_D2H(sig, d_sig, 64 * n);
    return KB_OK;
}
// plain staging: copy in, the three launches, copy out, all on the context's stream
int kb_signerset_sign_batch(kb_signerset* ss, size_t n, const uint32_t* key_idx, const uint8_t* nonces, const uint8_t* msg, const uint64_t* msg_off, uint8_t* sig)
{
    if (!ss) return KB_ERR_ARG;
    kb_ctx* ctx = ss->ctx;
    KB_ENTER();
    if ((ss->kind == KB_SIGNER_SCHNORR) != (nonces != nullptr)) return KB_ERR_ARG;
    if (n && (!key_idx || !msg_off || !sig)) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    uint32_t over = 0;
    for (size_t i = 0; i < n; i++) over |= (uint32_t)(key_idx[i] >= ss->nkeys);
    if (over) return KB_ERR_ARG;
    if (!kb_msg_off_ok(n, msg_off)) return KB_ERR_ARG;
    const size_t mbytes = (size_t)msg_off[n];
    if (mbytes && !msg) return KB_ERR_ARG;
    uint8_t* d_k = nullptr;
    if (nonces) KB_SCRATCH(6, 32 * n, d_k);
    const int rc = kb_signer_host_run(ss, n, key_idx, nonces, msg, msg_off, mbytes, sig, d_k);
    // the nonces do not outlive the call in scratch, on the error paths either
    if (d_k) cudaMemsetAsync(d_k, 0, 32 * n, ctx->stream);
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    KB_SYNC();
    return KB_OK;
}
}  // extern "C"
