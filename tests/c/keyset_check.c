/* tests/c/keyset_check.c — key sets used from plain C (no Python, no torch): create, verify, destroy.  Reads a fixture
 * written by tests/test_gpu_keyset.py::test_keyset_from_plain_c:
 *   u64 n, u64 msg_bytes, u64 nkeys, keys[32 nkeys], key_idx[u32 n], sig[64n], msg_off[u64 (n+1)], msg[msg_bytes],
 *   want_eddsa[n], want_schnorr[n]
 * and checks kb_keyset_verify_batch (schnorr = 0 and 1) against the expected statuses (which the Python side took from the
 * oracle), and that a key index outside the set and an empty key set are refused with KB_ERR_ARG.  Exit code 0 = all
 * equal. */
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

int main(int argc, char** argv)
{
    if (argc < 2) return 2;
    FILE* f = fopen(argv[1], "rb");
    if (!f) return 2;
    uint64_t hdr[3];
    if (fread(hdr, 8, 3, f) != 3) return 2;
    const size_t n = (size_t)hdr[0], mb = (size_t)hdr[1], nkeys = (size_t)hdr[2];
    uint8_t* keys = slurp(f, 32 * nkeys);
    uint32_t* idx = slurp(f, 4 * n);
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
    int bad = 0;
    kb_keyset* ks = NULL;
    bad += kb_keyset_create(ctx, 0, keys, &ks) != KB_ERR_ARG;
    rc = kb_keyset_create(ctx, nkeys, keys, &ks);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_keyset_create: %d %s\n", rc, kb_last_error(ctx));
        return 4;
    }
    uint8_t* st = malloc(n);
    for (int schnorr = 0; schnorr < 2; schnorr++) {
        memset(st, 0xAA, n);
        rc = kb_keyset_verify_batch(ks, n, idx, msg, off, sig, st, schnorr);
        if (rc != KB_OK) {
            fprintf(stderr, "kb_keyset_verify_batch: %d %s\n", rc, kb_last_error(ctx));
            return 4;
        }
        for (size_t i = 0; i < n; i++) bad += st[i] != want[schnorr][i];
    }
    if (n) {
        const uint32_t keep = idx[n - 1];
        idx[n - 1] = (uint32_t)nkeys;   /* outside the key set: refused before anything is launched */
        bad += kb_keyset_verify_batch(ks, n, idx, msg, off, sig, st, 0) != KB_ERR_ARG;
        idx[n - 1] = keep;
    }
    kb_keyset_destroy(ks);
    printf("keyset_check: n=%zu nkeys=%zu launches=%llu mismatches=%d\n", n, nkeys, (unsigned long long)kb_launch_count(ctx), bad);
    kb_ctx_destroy(ctx);
    free(st);
    return bad ? 1 : 0;
}
