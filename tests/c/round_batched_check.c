/* tests/c/round_batched_check.c — the batched share checks of a DKG round used from plain C (no Python, no torch).
 * Reads a fixture written by tests/test_gpu_round_batched.py::test_round_batched_from_plain_c:
 *   u64 n, u64 t, u64 ndealers, u64 wrong_dealers, commits[32 ndealers t], shares[32 m], want_verdict[m]   (m = ndealers n)
 * where want_verdict is what an EXACT context returns.  It checks that a new context is EXACT (no fallback count), that a
 * mode other than KB_ROUND_CHECK_EXACT / KB_ROUND_CHECK_BATCHED is refused with KB_ERR_ARG, and that a BATCHED round gives
 * the expected verdicts with one fallback per dealer that has a wrong share.  Exit code 0 = all as expected. */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

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
    uint64_t hdr[4];
    if (fread(hdr, 8, 4, f) != 4) return 2;
    const size_t n = (size_t)hdr[0], t = (size_t)hdr[1], nd = (size_t)hdr[2];
    const uint64_t wrong = hdr[3];
    const size_t m = nd * n;
    uint8_t* commits = slurp(f, 32 * nd * t);
    uint8_t* shares = slurp(f, 32 * m);
    uint8_t* want = slurp(f, m);
    fclose(f);
    uint8_t* v = malloc(m);
    kb_ctx* ctx = NULL;
    if (kb_ctx_create(0, &ctx) != KB_OK) return 3;
    int fails = 0;
    uint64_t fb = 99;
    if (kb_ctx_round_fallbacks(ctx, &fb) != KB_OK || fb != 0) fails++;
    if (kb_ctx_set_round_check(ctx, 2) != KB_ERR_ARG || kb_ctx_set_round_check(ctx, -1) != KB_ERR_ARG) fails++;
    if (kb_ctx_round_fallbacks(ctx, NULL) != KB_ERR_ARG) fails++;
    if (kb_ctx_set_round_check(ctx, KB_ROUND_CHECK_BATCHED) != KB_OK) fails++;
    size_t mismatches = 0;
    if (kb_dkg_verify_round(ctx, n, t, 0, nd, commits, shares, v) != KB_OK) {
        fprintf(stderr, "kb_dkg_verify_round: %s\n", kb_last_error(ctx));
        fails++;
    } else {
        for (size_t k = 0; k < m; k++) mismatches += v[k] != want[k];
    }
    if (kb_ctx_round_fallbacks(ctx, &fb) != KB_OK || fb != wrong) {
        fprintf(stderr, "fallbacks %llu, want %llu\n", (unsigned long long)fb, (unsigned long long)wrong);
        fails++;
    }
    kb_ctx_destroy(ctx);
    printf("mismatches=%zu fails=%d\n", mismatches, fails);
    free(commits);
    free(shares);
    free(want);
    free(v);
    return (mismatches == 0 && fails == 0) ? 0 : 1;
}
