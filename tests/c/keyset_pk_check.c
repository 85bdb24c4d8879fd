/* tests/c/keyset_pk_check.c — verification by public-key bytes from plain C (no Python, no torch).  Reads a fixture written
 * by tests/test_gpu_keyset_pk.py::test_pk_from_plain_c:
 *   u64 n, u64 msg_bytes, u64 nkeys, u64 hits, keys[32 nkeys], pk[32 n], sig[64 n], msg_off[u64 (n+1)], msg[msg_bytes],
 *   want_eddsa[n], want_schnorr[n]
 * and checks kb_keyset_verify_pk_batch and kb_mctx_keyset_verify_pk_batch (schnorr = 0 and 1) against the expected
 * statuses and hit count, and that a NULL key set and decreasing offsets are refused with KB_ERR_ARG.  The device form
 * (which needs device buffers, tested from Python) is called for its argument rules: n = 0 is KB_OK, a NULL key set or a
 * NULL buffer with n > 0 is KB_ERR_ARG.  Exit code 0 = all equal. */
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

static int count_bad(const uint8_t* st, const uint8_t* want, size_t n, uint64_t h, uint64_t hits)
{
    int bad = h != hits;
    for (size_t i = 0; i < n; i++) bad += st[i] != want[i];
    return bad;
}

int main(int argc, char** argv)
{
    if (argc < 2) return 2;
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    uint64_t hdr[4];
    if (fread(hdr, 8, 4, f) != 4) return 2;
    const size_t n = (size_t)hdr[0], mb = (size_t)hdr[1], nkeys = (size_t)hdr[2];
    const uint64_t hits = hdr[3];
    uint8_t* keys = slurp(f, 32 * nkeys);
    uint8_t* pk = slurp(f, 32 * n);
    uint8_t* sig = slurp(f, 64 * n);
    uint64_t* off = slurp(f, 8 * (n + 1));
    uint8_t* msg = slurp(f, mb);
    uint8_t* want[2];
    want[0] = slurp(f, n);
    want[1] = slurp(f, n);
    fclose(f);

    kb_ctx* ctx = NULL;
    int rc = kb_ctx_create(0, &ctx);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_ctx_create: %d (no GPU: there is no CPU fallback)\n", rc);
        return 3;
    }
    const int dev0 = 0;
    kb_mctx* m = NULL;
    kb_keyset* ks = NULL;
    kb_mkeyset* mks = NULL;
    if (kb_keyset_create(ctx, nkeys, keys, &ks) != KB_OK || kb_mctx_create(&dev0, 1, &m) != KB_OK || kb_mctx_keyset_create(m, nkeys, keys, &mks) != KB_OK) {
        fprintf(stderr, "key set creation failed: %s\n", kb_last_error(ctx));
        return 4;
    }
    int bad = 0;
    uint8_t* st = malloc(n);
    for (int schnorr = 0; schnorr < 2; schnorr++) {
        uint64_t h = 0;
        memset(st, 0xAA, n);
        rc = kb_keyset_verify_pk_batch(ks, n, pk, msg, off, sig, st, schnorr, &h);
        bad += rc != KB_OK || count_bad(st, want[schnorr], n, h, hits);
        memset(st, 0xAA, n);
        h = 0;
        rc = kb_mctx_keyset_verify_pk_batch(mks, n, pk, msg, off, sig, st, schnorr, &h);
        bad += rc != KB_OK || count_bad(st, want[schnorr], n, h, hits);
    }
    bad += kb_dev_keyset_verify_pk(ks, 0, NULL, NULL, NULL, NULL, NULL, 0, NULL, NULL) != KB_OK;
    bad += kb_dev_keyset_verify_pk(NULL, n, pk, msg, off, sig, st, 0, NULL, NULL) != KB_ERR_ARG;
    bad += kb_dev_keyset_verify_pk(ks, n, pk, msg, off, NULL, st, 0, NULL, NULL) != KB_ERR_ARG;
    bad += kb_keyset_verify_pk_batch(NULL, n, pk, msg, off, sig, st, 0, NULL) != KB_ERR_ARG;
    if (n > 1) {
        const uint64_t keep = off[1];
        off[1] = off[2] + 1;   /* decreasing offsets: refused before anything is launched */
        bad += kb_keyset_verify_pk_batch(ks, n, pk, msg, off, sig, st, 0, NULL) != KB_ERR_ARG;
        bad += kb_mctx_keyset_verify_pk_batch(mks, n, pk, msg, off, sig, st, 0, NULL) != KB_ERR_ARG;
        off[1] = keep;
    }
    kb_mctx_keyset_destroy(mks);
    kb_mctx_destroy(m);
    kb_keyset_destroy(ks);
    printf("keyset_pk_check: n=%zu nkeys=%zu hits=%llu launches=%llu mismatches=%d\n", n, nkeys, (unsigned long long)hits, (unsigned long long)kb_launch_count(ctx), bad);
    kb_ctx_destroy(ctx);
    free(st);
    return bad ? 1 : 0;
}
