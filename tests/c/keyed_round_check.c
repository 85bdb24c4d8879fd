/* tests/c/keyed_round_check.c — keyed DKG rounds and multi-device key sets used from plain C (no Python, no torch).
 * Reads a fixture written by tests/test_gpu_keyed_round.py::test_keyed_round_from_plain_c:
 *   u64 n, u64 t, u64 ndealers, u64 nkeys, u64 deal_msg_bytes, u64 resp_msg_bytes, keys[32 nkeys], commits[32 ndealers t],
 *   shares[32 m], deal_sig[64 m], deal_off[u64 (m+1)], deal_msg, resp_sig[64 m], resp_off[u64 (m+1)], resp_msg,
 *   want_verdict[m], want_deal[m], want_resp[m]                                               (m = ndealers n)
 * where the participants' keys serve as both dealers and verifiers.  It checks kb_dkg_process_round_keyed,
 * kb_mctx_keyset_verify_batch (the deals, key index k / n) and kb_mctx_dkg_process_round_keyed on a multi-device context
 * of device 0 against the expected bytes, and that a batch without a key set and a key index outside the set are refused
 * with KB_ERR_ARG.  Exit code 0 = all equal. */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "kyber_b200.h"

static void* slurp(FILE* f, size_t bytes)
{
    void* p = malloc(bytes ? bytes : 1);
    if (!p || fread(p, 1, bytes, f) != bytes) {
        fprintf(stderr, "short read\n");
        exit(2);
    }
    return p;
}

static int count_diff(const uint8_t* a, const uint8_t* b, size_t n)
{
    int d = 0;
    for (size_t i = 0; i < n; i++) d += a[i] != b[i];
    return d;
}

int main(int argc, char** argv)
{
    if (argc < 2) return 2;
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    uint64_t hdr[6];
    if (fread(hdr, 8, 6, f) != 6) return 2;
    const size_t n = (size_t)hdr[0], t = (size_t)hdr[1], nd = (size_t)hdr[2], nkeys = (size_t)hdr[3], dmb = (size_t)hdr[4], rmb = (size_t)hdr[5];
    const size_t m = nd * n;
    uint8_t* keys = slurp(f, 32 * nkeys);
    uint8_t* commits = slurp(f, 32 * nd * t);
    uint8_t* shares = slurp(f, 32 * m);
    uint8_t* dsig = slurp(f, 64 * m);
    uint64_t* doff = slurp(f, 8 * (m + 1));
    uint8_t* dmsg = slurp(f, dmb);
    uint8_t* rsig = slurp(f, 64 * m);
    uint64_t* roff = slurp(f, 8 * (m + 1));
    uint8_t* rmsg = slurp(f, rmb);
    uint8_t* want_v = slurp(f, m);
    uint8_t* want_d = slurp(f, m);
    uint8_t* want_r = slurp(f, m);
    fclose(f);
    uint8_t* v = malloc(m);
    uint8_t* ds = malloc(m);
    uint8_t* rs = malloc(m);
    uint32_t* idx = malloc(4 * m);
    for (size_t k = 0; k < m; k++) idx[k] = (uint32_t)(k / n);
    int bad = 0;

    /* one context */
    kb_ctx* ctx = NULL;
    int rc = kb_ctx_create(0, &ctx);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_ctx_create: %d (no GPU: there is no CPU fallback)\n", rc);
        return 3;
    }
    kb_keyset* ks = NULL;
    rc = kb_keyset_create(ctx, nkeys, keys, &ks);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_keyset_create: %d %s\n", rc, kb_last_error(ctx));
        return 4;
    }
    memset(v, 0xAA, m);
    memset(ds, 0xAA, m);
    memset(rs, 0xAA, m);
    rc = kb_dkg_process_round_keyed(ctx, ks, ks, n, t, 0, nd, KB_POINT_ENC32, commits, shares, v, dmsg, doff, dsig, ds, rmsg, roff, rsig, rs);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_dkg_process_round_keyed: %d %s\n", rc, kb_last_error(ctx));
        return 4;
    }
    bad += count_diff(v, want_v, m) + count_diff(ds, want_d, m) + count_diff(rs, want_r, m);
    /* a response batch without a verifier key set: refused before anything is launched */
    const uint64_t launches = kb_launch_count(ctx);
    bad += kb_dkg_process_round_keyed(ctx, ks, NULL, n, t, 0, nd, KB_POINT_ENC32, commits, shares, v, dmsg, doff, dsig, ds, rmsg, roff, rsig, rs) != KB_ERR_ARG;
    bad += kb_launch_count(ctx) != launches;
    kb_keyset_destroy(ks);
    kb_ctx_destroy(ctx);

    /* the multi-device context, here over device 0 */
    const int dev0 = 0;
    kb_mctx* mc = NULL;
    rc = kb_mctx_create(&dev0, 1, &mc);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_mctx_create: %d\n", rc);
        return 4;
    }
    kb_mkeyset* mk = NULL;
    bad += kb_mctx_keyset_create(mc, 0, keys, &mk) != KB_ERR_ARG;
    rc = kb_mctx_keyset_create(mc, nkeys, keys, &mk);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_mctx_keyset_create: %d %s\n", rc, kb_mctx_last_error(mc));
        return 4;
    }
    memset(ds, 0xAA, m);
    rc = kb_mctx_keyset_verify_batch(mk, m, idx, dmsg, doff, dsig, ds, 1);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_mctx_keyset_verify_batch: %d %s\n", rc, kb_mctx_last_error(mc));
        return 4;
    }
    bad += count_diff(ds, want_d, m);
    if (m) {
        idx[m - 1] = (uint32_t)nkeys;   /* outside the key set */
        bad += kb_mctx_keyset_verify_batch(mk, m, idx, dmsg, doff, dsig, ds, 1) != KB_ERR_ARG;
    }
    memset(v, 0xAA, m);
    memset(ds, 0xAA, m);
    memset(rs, 0xAA, m);
    rc = kb_mctx_dkg_process_round_keyed(mc, mk, mk, n, t, nd, KB_POINT_ENC32, commits, shares, v, dmsg, doff, dsig, ds, rmsg, roff, rsig, rs);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_mctx_dkg_process_round_keyed: %d %s\n", rc, kb_mctx_last_error(mc));
        return 4;
    }
    bad += count_diff(v, want_v, m) + count_diff(ds, want_d, m) + count_diff(rs, want_r, m);
    kb_mctx_keyset_destroy(mk);
    printf("keyed_round_check: n=%zu t=%zu ndealers=%zu nkeys=%zu launches=%llu mismatches=%d\n", n, t, nd, nkeys, (unsigned long long)kb_mctx_launch_count(mc), bad);
    kb_mctx_destroy(mc);
    free(v);
    free(ds);
    free(rs);
    free(idx);
    return bad ? 1 : 0;
}
