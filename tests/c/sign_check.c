/* tests/c/sign_check.c — signing used from plain C (no Python, no torch): kb_schnorr_sign_batch, then a Schnorr signer set
 * (create, kb_signerset_sign_batch, destroy).  Reads a fixture written by tests/test_gpu_sign.py::test_sign_from_plain_c:
 *   u64 n, u64 nkeys, keys[32 nkeys], key_idx[u32 n], nonces[32 n], msg_off[u64 n+1], msg[msg_off[n]], want_sig[64 n],
 *   want_pk[32 nkeys]
 * and checks both forms against the expected bytes (which the Python side took from kb_schnorr_sign_batch and
 * kb_point_mul_base_batch), and that a key index outside the set, a Schnorr set without nonces and a decreasing msg_off
 * are refused with KB_ERR_ARG while n = 0 is accepted.  Exit code 0 = all equal. */
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
    uint8_t* nonces = slurp(f, 32 * n);
    uint64_t* off = slurp(f, 8 * (n + 1));
    uint8_t* msg = slurp(f, (size_t)off[n]);
    uint8_t* want_sig = slurp(f, 64 * n);
    uint8_t* want_pk = slurp(f, 32 * nkeys);
    fclose(f);

    kb_ctx* ctx = NULL;
    int rc = kb_ctx_create(0, &ctx);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_ctx_create: %d (no GPU: there is no CPU fallback)\n", rc);
        return 3;
    }
    int bad = 0;
    uint8_t* x = malloc(32 * n + 1);
    uint8_t* sig = malloc(64 * n + 1);
    uint8_t* pk = malloc(32 * n + 32 * nkeys + 1);
    for (size_t i = 0; i < n; i++) memcpy(x + 32 * i, keys + 32 * (size_t)idx[i], 32);
    memset(sig, 0xAA, 64 * n);
    rc = kb_schnorr_sign_batch(ctx, n, x, nonces, msg, off, sig, pk);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_schnorr_sign_batch: %d %s\n", rc, kb_last_error(ctx));
        return 4;
    }
    for (size_t i = 0; i < n; i++) bad += memcmp(sig + 64 * i, want_sig + 64 * i, 64) != 0;
    for (size_t i = 0; i < n; i++) bad += memcmp(pk + 32 * i, want_pk + 32 * (size_t)idx[i], 32) != 0;

    kb_signerset* ss = NULL;
    rc = kb_signerset_create(ctx, nkeys, keys, KB_SIGNER_SCHNORR, pk, &ss);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_signerset_create: %d %s\n", rc, kb_last_error(ctx));
        return 4;
    }
    bad += memcmp(pk, want_pk, 32 * nkeys) != 0;
    memset(sig, 0xAA, 64 * n);
    rc = kb_signerset_sign_batch(ss, n, idx, nonces, msg, off, sig);
    if (rc != KB_OK) {
        fprintf(stderr, "kb_signerset_sign_batch: %d %s\n", rc, kb_last_error(ctx));
        return 4;
    }
    bad += memcmp(sig, want_sig, 64 * n) != 0;
    bad += kb_signerset_sign_batch(ss, n, idx, NULL, msg, off, sig) != KB_ERR_ARG;
    bad += kb_signerset_sign_batch(ss, 0, NULL, nonces, NULL, NULL, NULL) != KB_OK;
    bad += kb_schnorr_sign_batch(ctx, 0, NULL, NULL, NULL, NULL, NULL, NULL) != KB_OK;
    if (n > 1) {
        const uint32_t keep = idx[0];
        idx[0] = (uint32_t)nkeys;   /* outside the set: refused before anything is launched */
        bad += kb_signerset_sign_batch(ss, n, idx, nonces, msg, off, sig) != KB_ERR_ARG;
        idx[0] = keep;
        const uint64_t o1 = off[1];
        off[1] = off[2] + 1;        /* decreasing offsets */
        bad += kb_signerset_sign_batch(ss, n, idx, nonces, msg, off, sig) != KB_ERR_ARG;
        bad += kb_schnorr_sign_batch(ctx, n, x, nonces, msg, off, sig, NULL) != KB_ERR_ARG;
        off[1] = o1;
    }
    kb_signerset_destroy(ss);
    printf("sign_check: n=%zu nkeys=%zu launches=%llu mismatches=%d\n", n, nkeys, (unsigned long long)kb_launch_count(ctx), bad);
    kb_ctx_destroy(ctx);
    free(x);
    free(sig);
    free(pk);
    return bad ? 1 : 0;
}
