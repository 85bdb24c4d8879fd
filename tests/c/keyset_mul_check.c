/* tests/c/keyset_mul_check.c — keyed scalar multiplication used from plain C (no Python, no torch): create a key set,
 * kb_keyset_mul_batch, destroy.  Reads a fixture written by tests/test_gpu_keyset_mul.py::test_keyset_mul_from_plain_c:
 *   u64 n, u64 nkeys, keys[32 nkeys], key_idx[u32 n], scalars[32 n], want_out[32 n], want_status[n]
 * and checks kb_keyset_mul_batch with flags 0 and KB_FLAG_VARTIME against the expected bytes (which the Python side took
 * from kb_point_mul_batch), and that a key index outside the set and an unknown flag are refused with KB_ERR_ARG while
 * n = 0 is accepted.  Exit code 0 = all equal. */
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
    uint64_t hdr[2];
    if (fread(hdr, 8, 2, f) != 2) return 2;
    const size_t n = (size_t)hdr[0], nkeys = (size_t)hdr[1];
    uint8_t* keys = slurp(f, 32 * nkeys);
    uint32_t* idx = slurp(f, 4 * n);
    uint8_t* sc = slurp(f, 32 * n);
    uint8_t* want_out = slurp(f, 32 * n);
    uint8_t* want_st = slurp(f, n);
    fclose(f);

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
    int bad = 0;
    uint8_t* out = malloc(32 * n + 1);
    uint8_t* st = malloc(n + 1);
    const uint32_t flags[2] = {0, KB_FLAG_VARTIME};
    for (int k = 0; k < 2; k++) {
        memset(out, 0xAA, 32 * n);
        memset(st, 0xAA, n);
        rc = kb_keyset_mul_batch(ks, n, idx, sc, out, st, flags[k]);
        if (rc != KB_OK) {
            fprintf(stderr, "kb_keyset_mul_batch: %d %s\n", rc, kb_last_error(ctx));
            return 4;
        }
        for (size_t i = 0; i < n; i++) bad += (st[i] != want_st[i]) + (memcmp(out + 32 * i, want_out + 32 * i, 32) != 0);
    }
    bad += kb_keyset_mul_batch(ks, n, idx, sc, out, st, KB_FLAG_SHARED_POINT) != KB_ERR_ARG;
    bad += kb_keyset_mul_batch(ks, 0, NULL, NULL, NULL, NULL, 0) != KB_OK;
    if (n) {
        const uint32_t keep = idx[0];
        idx[0] = (uint32_t)nkeys;   /* outside the key set: refused before anything is launched */
        bad += kb_keyset_mul_batch(ks, n, idx, sc, out, st, 0) != KB_ERR_ARG;
        idx[0] = keep;
    }
    kb_keyset_destroy(ks);
    printf("keyset_mul_check: n=%zu nkeys=%zu launches=%llu mismatches=%d\n", n, nkeys, (unsigned long long)kb_launch_count(ctx), bad);
    kb_ctx_destroy(ctx);
    free(out);
    free(st);
    return bad ? 1 : 0;
}
