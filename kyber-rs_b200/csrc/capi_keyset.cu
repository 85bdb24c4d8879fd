// capi_keyset.cu — key sets: EdDSA / Schnorr verification under registered public keys (include/kyber_b200.h)
#define KB_K_KEYSET
// the field-arithmetic bodies of the other verifiers (capi_verify.cu): k_keyset_verify is a verifier of the same kind
#define KB_FE_MUL_RIP
#define KB_FE_SQ_RIP
#define KB_FE_SUBMASK
#include <random>
#include <vector>

#include "ctx.cuh"
#include "kernels.cuh"

// One allocation per key set: the combs (KB_KEY_ENTRIES affine entries per key), then the 32-byte keys, then one byte of
// facts per key.  It is not part of the context's scratch, so kb_ctx_wipe leaves it alone.
// A second, small allocation holds the lookup table of kb_dev_keyset_verify_pk: open addressing with linear probing, one
// key index per slot (KB_PK_MISS: empty), hmask + 1 >= 2 nkeys slots, hashed with kb_pk_hash under a seed drawn for this
// set (a fixed hash would let whoever chooses the queried pks aim them at long runs).  hprobe is the longest run any
// registered key needed; a lookup reads at most that many slots.
struct kb_keyset {
    kb_ctx* ctx;
    size_t nkeys;
    void* mem;
    ge_precomp* table;
    uint8_t* pk;
    uint8_t* facts;
    uint32_t* htab;
    uint32_t hmask, hprobe;
    uint64_t hseed[2];
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

// the lookup table of the host keys pk[0 .. nkeys) (see kb_keyset), copied to ks->htab; a key whose bytes repeat an
// earlier key's is not inserted, so a lookup finds the lowest index of equal bytes
static int kb_keyset_build_lookup(kb_keyset* ks, const uint8_t* pk)
{
    kb_ctx* ctx = ks->ctx;
    const size_t nkeys = ks->nkeys;
    if (nkeys > ((size_t)1 << 31)) return KB_ERR_NOMEM;
    size_t cap = 2;
    while (cap < 2 * nkeys) cap <<= 1;
    std::random_device rd;
    for (int k = 0; k < 2; k++) ks->hseed[k] = ((uint64_t)rd() << 32) ^ (uint64_t)rd();
    ks->hmask = (uint32_t)(cap - 1);
    ks->hprobe = 0;
    std::vector<uint32_t> tab(cap, KB_PK_MISS);
    for (size_t k = 0; k < nkeys; k++) {
        uint32_t w[8];
        memcpy(w, pk + 32 * k, 32);   // little-endian words, as kb_load32 reads them on the device
        const uint64_t h = kb_pk_hash(w, ks->hseed[0], ks->hseed[1]);
        for (uint32_t p = 0;; p++) {
            uint32_t& e = tab[kb_pk_slot(h, p, ks->hmask)];
            if (e == KB_PK_MISS) {
                e = (uint32_t)k;
                if (p + 1 > ks->hprobe) ks->hprobe = p + 1;
                break;
            }
            if (memcmp(pk + 32 * (size_t)e, pk + 32 * k, 32) == 0) break;
        }
    }
    cudaError_t e = cudaMalloc(&ks->htab, 4 * cap);
    if (e != cudaSuccess) {
        kb_fail(ctx, e, "kb_keyset_create: cudaMalloc of the lookup table");
        return KB_ERR_NOMEM;
    }
    e = cudaMemcpy(ks->htab, tab.data(), 4 * cap, cudaMemcpyHostToDevice);
    return e == cudaSuccess ? KB_OK : kb_fail(ctx, e, "kb_keyset_create: copy of the lookup table");
}

// Scratch of kb_dev_keyset_verify_pk: kidx[n], hit_item[n], hit_key[n], miss_item[n], the per-block counts, then
// {hits, misses}
#define KB_SLOT_PK_PART 54
// the launches of kb_dev_keyset_verify_pk; every grid is sized for n and every kernel after the scan reads its count from
// the device, so nothing waits for the host
static int kb_keyset_pk_launch(kb_keyset* ks, size_t n, const uint8_t* d_pk, const uint8_t* d_msg, const uint64_t* d_msg_off, const uint8_t* d_sig, uint8_t* d_status, int schnorr,
                               unsigned long long* d_hits, cudaStream_t st)
{
    kb_ctx* ctx = ks->ctx;
    const uint32_t nblk = kb_blocks(n, KB_PK_BLOCK);
    uint32_t *part, *xyz;
    uint8_t* fl;
    KB_SCRATCH(KB_SLOT_PK_PART, 4 * (4 * n + nblk + 2), part);
    KB_SCRATCH(KB_SLOT_XYZ, KB_VERIFY_SCRATCH_BYTES * n, xyz);
    KB_SCRATCH(KB_SLOT_FLAGS, KB_VERIFY_FLAG_BYTES(n), fl);
    uint32_t *kidx = part, *hit_item = part + n, *hit_key = part + 2 * n, *miss_item = part + 3 * n, *blk = part + 4 * n, *cnt = blk + nblk;
    k_pk_lookup<<<nblk, KB_PK_BLOCK, 0, st>>>(n, d_pk, ks->htab, ks->hmask, ks->hprobe, ks->hseed[0], ks->hseed[1], ks->pk, kidx, blk);
    KB_LAUNCHED();
    k_pk_scan<<<1, 1024, 0, st>>>(n, nblk, blk, cnt, d_hits);
    KB_LAUNCHED();
    k_pk_scatter<<<nblk, KB_PK_BLOCK, 0, st>>>(n, kidx, blk, hit_item, hit_key, miss_item);
    KB_LAUNCHED();
    // hits: the comb path of kb_dev_keyset_verify, 96 bytes of xyz and one flag byte per slot
    const unsigned g1 = kb_blocks(n, KB_THREADS), g2 = kb_blocks((n + KB_INV_K - 1) / KB_INV_K, KB_THREADS);
    if (schnorr) k_keyset_verify_pk<true><<<g1, KB_THREADS, 0, st>>>(cnt, hit_item, hit_key, ks->pk, ks->facts, ks->table, d_msg, d_msg_off, d_sig, ctx->comb, xyz, fl);
    else k_keyset_verify_pk<false><<<g1, KB_THREADS, 0, st>>>(cnt, hit_item, hit_key, ks->pk, ks->facts, ks->table, d_msg, d_msg_off, d_sig, ctx->comb, xyz, fl);
    KB_LAUNCHED();
    if (schnorr) k_verify_stage2_list<true><<<g2, KB_THREADS, 0, st>>>(cnt, hit_item, xyz, fl, d_sig, d_status);
    else k_verify_stage2_list<false><<<g2, KB_THREADS, 0, st>>>(cnt, hit_item, xyz, fl, d_sig, d_status);
    KB_LAUNCHED();
    // misses: the default half-size-scalar path of kb_verify_launch (whatever KB_VERIFY_FULL / KB_VERIFY_SPLIT say: the
    // statuses are the same), its records in xyz after the hits are done with it
    const uint32_t* mcnt = cnt + 1;
    const unsigned th = kb_item_threads(ctx, n);
    if (schnorr) k_verify_half_prep_list<true><<<g1, KB_THREADS, 0, st>>>(n, mcnt, miss_item, d_pk, d_msg, d_msg_off, d_sig, xyz);
    else k_verify_half_prep_list<false><<<g1, KB_THREADS, 0, st>>>(n, mcnt, miss_item, d_pk, d_msg, d_msg_off, d_sig, xyz);
    KB_LAUNCHED();
    const uint32_t* perm = nullptr;
#if KB_HALF_JOINT
    // sorted or not by the rule of kb_verify_launch, applied to the upper bound n
    if (ctx->verify_sort && (n >= 16384 || ctx->verify_sort == 2)) {
        uint32_t* pm = reinterpret_cast<uint32_t*>(fl);
        uint8_t* keys = fl + 4 * n;
        uint32_t* hist = reinterpret_cast<uint32_t*>(fl + ((5 * n + 255) & ~(size_t)255));
        KB_CUDA(cudaMemsetAsync(hist, 0, 4 * KB_SORT_BINS, st));
        k_half_sort_count_list<<<kb_blocks(n, 256), 256, 0, st>>>(mcnt, xyz, keys, hist);
        KB_LAUNCHED();
        k_half_sort_scan<<<1, 32, 0, st>>>(hist, hist + KB_SORT_BINS);
        KB_LAUNCHED();
        k_half_sort_scatter_list<<<kb_blocks(n, 256), 256, 0, st>>>(mcnt, keys, hist + KB_SORT_BINS, pm);
        KB_LAUNCHED();
        perm = pm;
    }
#endif
    if (schnorr) k_verify_half_main_list<true><<<kb_blocks(n, th), th, 0, st>>>(n, mcnt, miss_item, xyz, perm, d_status, ctx->comb, ctx->verify_min_windows, ctx->verify_force_redo);
    else k_verify_half_main_list<false><<<kb_blocks(n, th), th, 0, st>>>(n, mcnt, miss_item, xyz, perm, d_status, ctx->comb, ctx->verify_min_windows, ctx->verify_force_redo);
    KB_LAUNCHED();
    return KB_OK;
}

// ---- keyed DKG rounds: the signer of every deal and response is implied by the item's position in the round
// The argument checks of both forms, made before anything is launched: every key a batch names is in its key set, and
// each key set belongs to ctx.
static bool kb_keyed_round_ok(const kb_ctx* ctx, const kb_keyset* dealers, const kb_keyset* verifiers, size_t n, size_t dealer_hi, const void* deal_sig, const void* resp_sig)
{
    if ((deal_sig && !dealers) || (resp_sig && !verifiers)) return false;
    if (dealers && (dealers->ctx != ctx || dealers->nkeys < dealer_hi)) return false;
    if (verifiers && (verifiers->ctx != ctx || verifiers->nkeys < n)) return false;
    return true;
}
// one Schnorr batch of m items on device buffers (deal: signer dealer_lo + k / n, response: signer k % n); xyz (96 B per
// item) and fl (1 B) are scratch
static int kb_keyed_round_launch(kb_ctx* ctx, const kb_keyset* ks, bool resp, size_t m, size_t n, size_t dealer_lo, const uint8_t* d_msg, const uint64_t* d_msg_off, uint64_t msg_base,
                                 const uint8_t* d_sig, uint8_t* d_status, uint32_t* xyz, uint8_t* fl, cudaStream_t st)
{
    const unsigned g1 = kb_blocks(m, KB_THREADS), g2 = kb_blocks((m + KB_INV_K - 1) / KB_INV_K, KB_THREADS);
    if (resp) k_keyset_verify_round<true><<<g1, KB_THREADS, 0, st>>>(m, n, 0, ks->pk, ks->facts, ks->table, d_msg, d_msg_off, msg_base, d_sig, ctx->comb, xyz, fl);
    else k_keyset_verify_round<false><<<g1, KB_THREADS, 0, st>>>(m, n, dealer_lo, ks->pk, ks->facts, ks->table, d_msg, d_msg_off, msg_base, d_sig, ctx->comb, xyz, fl);
    KB_LAUNCHED();
    k_verify_stage2<true><<<g2, KB_THREADS, 0, st>>>(m, xyz, fl, d_sig, d_status);
    KB_LAUNCHED();
    return KB_OK;
}
// pointers and message offsets of one host batch of m items
static bool kb_keyed_batch_ok(size_t m, const uint8_t* msg, const uint64_t* msg_off, uint8_t* status)
{
    if (m == 0) return true;
    if (!msg_off || !status || !kb_msg_off_ok(m, msg_off)) return false;
    return msg_off[m] == msg_off[0] || msg;
}
// plain staging of one host batch on the context's stream: only msg[msg_off[0] .. msg_off[m]) is copied
static int kb_keyed_batch_host(kb_ctx* ctx, const kb_keyset* ks, bool resp, size_t m, size_t n, size_t dealer_lo, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status)
{
    if (m == 0) return KB_OK;
    const uint64_t m0 = msg_off[0];
    const size_t mbytes = (size_t)(msg_off[m] - m0);
    uint8_t *d_sig, *d_m, *d_st, *fl;
    uint64_t* d_off;
    uint32_t* xyz;
    KB_SCRATCH(1, 64 * m, d_sig);
    KB_SCRATCH(2, mbytes, d_m);
    KB_SCRATCH(3, 8 * (m + 1), d_off);
    KB_SCRATCH(4, m, d_st);
    KB_SCRATCH(KB_SLOT_XYZ, 96 * m, xyz);
    KB_SCRATCH(KB_SLOT_FLAGS, m, fl);
    KB_H2D(d_sig, sig, 64 * m);
    if (mbytes) KB_H2D(d_m, msg + m0, mbytes);
    KB_H2D(d_off, msg_off, 8 * (m + 1));
    const int rc = kb_keyed_round_launch(ctx, ks, resp, m, n, dealer_lo, d_m, d_off, m0, d_sig, d_st, xyz, fl, ctx->stream);
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    KB_D2H(status, d_st, m);
    KB_SYNC();
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
    if (rc == KB_OK) rc = kb_keyset_build_lookup(ks, pk);
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
    if (ks->htab) cudaFree(ks->htab);
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

// ---- verification by public-key bytes: registered keys on the comb path, every other key on the general verifier
int kb_dev_keyset_verify_pk(kb_keyset* ks, size_t n, const void* d_pk, const void* d_msg, const void* d_msg_off, const void* d_sig, void* d_status, int schnorr, void* d_hits, void* stream)
{
    if (!ks) return KB_ERR_ARG;
    kb_ctx* ctx = ks->ctx;
    if (n && (!d_pk || !d_msg_off || !d_sig || !d_status)) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    if (n > UINT32_MAX) return KB_ERR_ARG;   // item numbers are 32-bit in the sub-batch lists
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    KB_DEV_RETURN(st, kb_keyset_pk_launch(ks, n, (const uint8_t*)d_pk, (const uint8_t*)d_msg, (const uint64_t*)d_msg_off, (const uint8_t*)d_sig, (uint8_t*)d_status, schnorr,
                                          (unsigned long long*)d_hits, st));
}
// plain staging: copy in, the device form, copy out, all on the context's stream
int kb_keyset_verify_pk_batch(kb_keyset* ks, size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status, int schnorr, uint64_t* hits)
{
    if (!ks) return KB_ERR_ARG;
    kb_ctx* ctx = ks->ctx;
    KB_ENTER();
    if (n && (!pk || !msg_off || !sig || !status)) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    if (n > UINT32_MAX || !kb_msg_off_ok(n, msg_off)) return KB_ERR_ARG;
    const size_t mbytes = (size_t)msg_off[n];
    if (mbytes && !msg) return KB_ERR_ARG;
    uint8_t *d_pk, *d_sig, *d_m, *d_st;
    uint64_t *d_off, *d_hits;
    KB_SCRATCH(0, 32 * n, d_pk);
    KB_SCRATCH(1, 64 * n, d_sig);
    KB_SCRATCH(2, mbytes, d_m);
    KB_SCRATCH(3, 8 * (n + 1), d_off);
    KB_SCRATCH(4, n, d_st);
    KB_SCRATCH(5, 8, d_hits);
    KB_H2D(d_pk, pk, 32 * n);
    KB_H2D(d_sig, sig, 64 * n);
    if (mbytes) KB_H2D(d_m, msg, mbytes);
    KB_H2D(d_off, msg_off, 8 * (n + 1));
    const int rc = kb_dev_keyset_verify_pk(ks, n, d_pk, d_m, d_off, d_sig, d_st, schnorr, d_hits, ctx->stream);
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    uint64_t h = 0;
    KB_D2H(status, d_st, n);
    KB_D2H(&h, d_hits, 8);
    KB_SYNC();
    if (hits) *hits = h;
    return KB_OK;
}

// ---- Point::mul(s, Some(keys[key_idx[i]])): k_keyset_mul, then the batch compression of kb_dev_point_mul
int kb_dev_keyset_mul(kb_keyset* ks, size_t n, const void* d_key_idx, const void* d_scalars, void* d_out, void* d_status, uint32_t flags, void* stream)
{
    if (!ks) return KB_ERR_ARG;
    kb_ctx* ctx = ks->ctx;
    if ((flags & ~KB_FLAG_VARTIME) || (n && (!d_key_idx || !d_scalars || !d_out))) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    uint32_t* xyz;
    uint8_t* bad = (uint8_t*)d_status;
    KB_SCRATCH(KB_SLOT_XYZ, 96 * n, xyz);
    if (!bad) KB_SCRATCH(KB_SLOT_FLAGS, n, bad);
    const unsigned th = kb_item_threads(ctx, n);
    const uint32_t* idx = (const uint32_t*)d_key_idx;
    const uint8_t* sc = (const uint8_t*)d_scalars;
    if (flags & KB_FLAG_VARTIME)
        k_keyset_mul<false><<<kb_blocks(n, th), th, 0, st>>>(n, idx, ks->nkeys, ks->pk, ks->facts, ks->table, sc, xyz, bad);
    else
        k_keyset_mul<true><<<kb_blocks(n, th), th, 0, st>>>(n, idx, ks->nkeys, ks->pk, ks->facts, ks->table, sc, xyz, bad);
    KB_LAUNCHED();
    k_compress_batch<<<kb_blocks((n + KB_INV_K - 1) / KB_INV_K, KB_THREADS), KB_THREADS, 0, st>>>(n, xyz, bad, (uint8_t*)d_out);
    KB_LAUNCHED();
    KB_DEV_RETURN(st, KB_OK);
}
// plain staging as kb_point_mul_batch: copy in, the two launches, copy out, all on the context's stream
int kb_keyset_mul_batch(kb_keyset* ks, size_t n, const uint32_t* key_idx, const uint8_t* scalars, uint8_t* out, uint8_t* status, uint32_t flags)
{
    if (!ks) return KB_ERR_ARG;
    kb_ctx* ctx = ks->ctx;
    KB_ENTER();
    if ((flags & ~KB_FLAG_VARTIME) || (n && (!key_idx || !scalars || !out))) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    uint32_t over = 0;
    for (size_t i = 0; i < n; i++) over |= (uint32_t)(key_idx[i] >= ks->nkeys);
    if (over) return KB_ERR_ARG;
    uint8_t *d_s, *d_o, *d_st;
    uint32_t* d_idx;
    KB_SCRATCH(0, 32 * n, d_s);
    KB_SCRATCH(1, 32 * n, d_o);
    KB_SCRATCH(2, 4 * n, d_idx);
    KB_SCRATCH(3, n, d_st);
    KB_H2D(d_s, scalars, 32 * n);
    KB_H2D(d_idx, key_idx, 4 * n);
    const int rc = kb_dev_keyset_mul(ks, n, d_idx, d_s, d_o, d_st, flags, ctx->stream);
    // scalars that are not declared public (KB_FLAG_VARTIME) do not outlive the call in device scratch
    if (!(flags & KB_FLAG_VARTIME)) KB_CUDA(cudaMemsetAsync(d_s, 0, 32 * n, ctx->stream));
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    KB_D2H(out, d_o, 32 * n);
    if (status) KB_D2H(status, d_st, n);
    KB_SYNC();
    return KB_OK;
}

int kb_dev_dkg_process_round_keyed(kb_ctx* ctx, const kb_keyset* dealers, const kb_keyset* verifiers, size_t n, size_t t, size_t dealer_lo, size_t ndealers, int fmt, const void* d_commits,
                                   const void* d_shares, void* d_verdict, const void* d_deal_msg, const void* d_deal_msg_off, const void* d_deal_sig, void* d_deal_status,
                                   const void* d_resp_msg, const void* d_resp_msg_off, const void* d_resp_sig, void* d_resp_status, void* stream)
{
    if (!ctx || !t || (fmt != KB_POINT_ENC32 && fmt != KB_POINT_LIMBS40) || (n && ndealers && (!d_commits || !d_shares || !d_verdict))) return KB_ERR_ARG;
    if (d_deal_sig && (!d_deal_msg_off || !d_deal_status)) return KB_ERR_ARG;
    if (d_resp_sig && (!d_resp_msg_off || !d_resp_status)) return KB_ERR_ARG;
    if (ndealers > SIZE_MAX - dealer_lo || !kb_keyed_round_ok(ctx, dealers, verifiers, n, dealer_lo + ndealers, d_deal_sig, d_resp_sig)) return KB_ERR_ARG;
    const size_t m = n * ndealers;
    if (m == 0) return KB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    int rc = kb_dkg_round_run(ctx, n, t, ndealers, d_commits, fmt == KB_POINT_LIMBS40, (const uint8_t*)d_shares, (uint8_t*)d_verdict, st);
    if (rc != KB_OK) return rc;
    uint32_t* xyz;
    uint8_t* fl;
    KB_SCRATCH(KB_SLOT_XYZ, 96 * m, xyz);
    KB_SCRATCH(KB_SLOT_FLAGS, m, fl);
    if (d_deal_sig) {
        rc = kb_keyed_round_launch(ctx, dealers, false, m, n, dealer_lo, (const uint8_t*)d_deal_msg, (const uint64_t*)d_deal_msg_off, 0, (const uint8_t*)d_deal_sig, (uint8_t*)d_deal_status, xyz, fl, st);
        if (rc != KB_OK) return rc;
    }
    if (d_resp_sig) {
        rc = kb_keyed_round_launch(ctx, verifiers, true, m, n, 0, (const uint8_t*)d_resp_msg, (const uint64_t*)d_resp_msg_off, 0, (const uint8_t*)d_resp_sig, (uint8_t*)d_resp_status, xyz, fl, st);
        if (rc != KB_OK) return rc;
    }
    KB_DEV_RETURN(st, KB_OK);
}
int kb_dkg_process_round_keyed(kb_ctx* ctx, const kb_keyset* dealers, const kb_keyset* verifiers, size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, int fmt, const void* commits,
                               const uint8_t* shares, uint8_t* verdict, const uint8_t* deal_msg, const uint64_t* deal_msg_off, const uint8_t* deal_sig, uint8_t* deal_status,
                               const uint8_t* resp_msg, const uint64_t* resp_msg_off, const uint8_t* resp_sig, uint8_t* resp_status)
{
    if (!ctx || dealer_hi < dealer_lo || (fmt != KB_POINT_ENC32 && fmt != KB_POINT_LIMBS40)) return KB_ERR_ARG;
    if (!kb_keyed_round_ok(ctx, dealers, verifiers, n, dealer_hi, deal_sig, resp_sig)) return KB_ERR_ARG;
    // the signature arrays hold the m = (dealer_hi - dealer_lo) * n items of this dealer range, item (d - dealer_lo) * n + i
    const size_t m = (dealer_hi - dealer_lo) * n;
    if (deal_sig && !kb_keyed_batch_ok(m, deal_msg, deal_msg_off, deal_status)) return KB_ERR_ARG;
    if (resp_sig && !kb_keyed_batch_ok(m, resp_msg, resp_msg_off, resp_status)) return KB_ERR_ARG;
    int rc;
    if (fmt == KB_POINT_LIMBS40) rc = kb_dkg_verify_round_limbs(ctx, n, t, dealer_lo, dealer_hi, (const int32_t*)commits, shares, verdict);
    else rc = kb_dkg_verify_round(ctx, n, t, dealer_lo, dealer_hi, (const uint8_t*)commits, shares, verdict);
    if (rc != KB_OK) return rc;
    if (deal_sig) {
        rc = kb_keyed_batch_host(ctx, dealers, false, m, n, dealer_lo, deal_msg, deal_msg_off, deal_sig, deal_status);
        if (rc != KB_OK) return rc;
    }
    if (resp_sig) rc = kb_keyed_batch_host(ctx, verifiers, true, m, n, 0, resp_msg, resp_msg_off, resp_sig, resp_status);
    return rc;
}
}  // extern "C"
