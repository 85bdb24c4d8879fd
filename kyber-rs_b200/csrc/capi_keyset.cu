// capi_keyset.cu — key sets: EdDSA / Schnorr verification under registered public keys (include/kyber_b200.h)
#define KB_K_KEYSET
// the field-arithmetic bodies of the other verifiers (capi_verify.cu): k_keyset_verify is a verifier of the same kind
#define KB_FE_MUL_RIP
#define KB_FE_SQ_RIP
#define KB_FE_SUBMASK
#include "ctx.cuh"
#include "kernels.cuh"

// One allocation per key set: the combs (KB_KEY_ENTRIES affine entries per key), then the 32-byte keys, then one byte of
// facts per key.  It is not part of the context's scratch, so kb_ctx_wipe leaves it alone.
struct kb_keyset {
    kb_ctx* ctx;
    size_t nkeys;
    void* mem;
    ge_precomp* table;
    uint8_t* pk;
    uint8_t* facts;
};
#define KB_KEY_TABLE_BYTES (sizeof(ge_precomp) * (size_t)KB_KEY_ENTRIES)
static_assert(KB_KEY_TABLE_BYTES == 393216, "384 KiB of comb per key");

// k_keyset_verify, k_verify_stage2, k_keyset_bad_index on device buffers; xyz (96 B per item) and fl (1 B) are scratch
static int kb_keyset_launch(kb_keyset* ks, size_t n, const uint32_t* d_key_idx, const uint8_t* d_msg, const uint64_t* d_msg_off, const uint8_t* d_sig, uint8_t* d_status, int schnorr,
                            uint32_t* xyz, uint8_t* fl, cudaStream_t st)
{
    kb_ctx* ctx = ks->ctx;
    const unsigned g1 = kb_blocks(n, KB_THREADS), g2 = kb_blocks((n + KB_INV_K - 1) / KB_INV_K, KB_THREADS);
    if (schnorr) k_keyset_verify<true><<<g1, KB_THREADS, 0, st>>>(n, d_key_idx, ks->nkeys, ks->pk, ks->facts, ks->table, d_msg, d_msg_off, d_sig, ctx->comb, xyz, fl);
    else k_keyset_verify<false><<<g1, KB_THREADS, 0, st>>>(n, d_key_idx, ks->nkeys, ks->pk, ks->facts, ks->table, d_msg, d_msg_off, d_sig, ctx->comb, xyz, fl);
    KB_LAUNCHED();
    if (schnorr) k_verify_stage2<true><<<g2, KB_THREADS, 0, st>>>(n, xyz, fl, d_sig, d_status);
    else k_verify_stage2<false><<<g2, KB_THREADS, 0, st>>>(n, xyz, fl, d_sig, d_status);
    KB_LAUNCHED();
    k_keyset_bad_index<<<kb_blocks(n, 256), 256, 0, st>>>(n, d_key_idx, ks->nkeys, d_status);
    KB_LAUNCHED();
    return KB_OK;
}

extern "C" {
int kb_keyset_create(kb_ctx* ctx, size_t nkeys, const uint8_t* pk, kb_keyset** out)
{
    KB_ENTER();
    if (!out) return KB_ERR_ARG;
    *out = nullptr;
    if (nkeys == 0 || !pk) return KB_ERR_ARG;
    const size_t per_key = KB_KEY_TABLE_BYTES + 32 + 1;
    if (nkeys > (SIZE_MAX - 256) / per_key) return KB_ERR_NOMEM;
    kb_keyset* ks = (kb_keyset*)calloc(1, sizeof(kb_keyset));
    if (!ks) return KB_ERR_NOMEM;
    ks->ctx = ctx;
    ks->nkeys = nkeys;
    const cudaError_t e = cudaMalloc(&ks->mem, nkeys * per_key);
    if (e != cudaSuccess) {
        kb_fail(ctx, e, "kb_keyset_create: cudaMalloc of the key combs");
        free(ks);
        return KB_ERR_NOMEM;
    }
    ks->table = reinterpret_cast<ge_precomp*>(ks->mem);
    ks->pk = reinterpret_cast<uint8_t*>(ks->mem) + nkeys * KB_KEY_TABLE_BYTES;   // 16-byte aligned: the comb is 384 KiB per key
    ks->facts = ks->pk + 32 * nkeys;
    int rc = KB_OK;
    const cudaError_t ce = cudaMemcpyAsync(ks->pk, pk, 32 * nkeys, cudaMemcpyHostToDevice, ctx->stream);
    if (ce != cudaSuccess) {
        rc = kb_fail(ctx, ce, "kb_keyset_create: copy of the keys");
    } else {
        k_keyset_build<<<kb_blocks(nkeys * KB_KEY_POS, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(nkeys, ks->pk, ks->facts, ks->table);
        ctx->launches++;
        cudaError_t le = cudaGetLastError();
        if (le == cudaSuccess) le = cudaStreamSynchronize(ctx->stream);
        if (le != cudaSuccess) rc = kb_fail(ctx, le, "kb_keyset_create: k_keyset_build");
    }
    if (rc != KB_OK) {
        kb_keyset_destroy(ks);
        return rc;
    }
    *out = ks;
    return KB_OK;
}
void kb_keyset_destroy(kb_keyset* ks)
{
    if (!ks) return;
    cudaSetDevice(ks->ctx->device);
    cudaDeviceSynchronize();   // verify calls on any stream may still read the combs
    if (ks->mem) cudaFree(ks->mem);
    free(ks);
}
int kb_dev_keyset_verify(kb_keyset* ks, size_t n, const void* d_key_idx, const void* d_msg, const void* d_msg_off, const void* d_sig, void* d_status, int schnorr, void* stream)
{
    if (!ks) return KB_ERR_ARG;
    kb_ctx* ctx = ks->ctx;
    if (n && (!d_key_idx || !d_msg_off || !d_sig || !d_status)) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    uint32_t* xyz;
    uint8_t* fl;
    KB_SCRATCH(KB_SLOT_XYZ, 96 * n, xyz);
    KB_SCRATCH(KB_SLOT_FLAGS, n, fl);
    KB_DEV_RETURN(st, kb_keyset_launch(ks, n, (const uint32_t*)d_key_idx, (const uint8_t*)d_msg, (const uint64_t*)d_msg_off, (const uint8_t*)d_sig, (uint8_t*)d_status, schnorr, xyz, fl, st));
}
// plain staging: copy in, the three launches, copy out, all on the context's stream
int kb_keyset_verify_batch(kb_keyset* ks, size_t n, const uint32_t* key_idx, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status, int schnorr)
{
    if (!ks) return KB_ERR_ARG;
    kb_ctx* ctx = ks->ctx;
    KB_ENTER();
    if (n && (!key_idx || !msg_off || !sig || !status)) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    uint32_t over = 0;
    for (size_t i = 0; i < n; i++) over |= (uint32_t)(key_idx[i] >= ks->nkeys);
    if (over) return KB_ERR_ARG;
    if (!kb_msg_off_ok(n, msg_off)) return KB_ERR_ARG;
    const size_t mbytes = (size_t)msg_off[n];
    if (mbytes && !msg) return KB_ERR_ARG;
    uint32_t* d_idx;
    uint8_t *d_sig, *d_m, *d_st;
    uint64_t* d_off;
    KB_SCRATCH(0, 4 * n, d_idx);
    KB_SCRATCH(1, 64 * n, d_sig);
    KB_SCRATCH(2, mbytes, d_m);
    KB_SCRATCH(3, 8 * (n + 1), d_off);
    KB_SCRATCH(4, n, d_st);
    KB_H2D(d_idx, key_idx, 4 * n);
    KB_H2D(d_sig, sig, 64 * n);
    if (mbytes) KB_H2D(d_m, msg, mbytes);
    KB_H2D(d_off, msg_off, 8 * (n + 1));
    const int rc = kb_dev_keyset_verify(ks, n, d_idx, d_m, d_off, d_sig, d_st, schnorr, ctx->stream);
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    KB_D2H(status, d_st, n);
    KB_SYNC();
    return KB_OK;
}
}  // extern "C"
