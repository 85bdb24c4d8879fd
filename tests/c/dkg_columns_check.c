/* tests/c/dkg_columns_check.c — the share checks of a verifier range used from plain C (no Python, no torch).
 * Reads a fixture written by tests/test_gpu_dkg_columns.py::test_columns_from_plain_c:
 *   u64 n, u64 t, u64 ndealers, u64 ver_lo, u64 ver_hi, commits[32 ndealers t], shares[32 m], want_verdict[m]
 * (m = ndealers (ver_hi - ver_lo)), where want_verdict is what kb_vss_verify_deals_batch returns on the same items.  It checks
 * the verdicts in both round-check modes with a fallback count of 0, the argument errors, and that an empty dealer range
 * returns KB_OK.  Exit code 0 = all as expected. */
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
    uint64_t hdr[5];
    if (fread(hdr, 8, 5, f) != 5) return 2;
    const size_t n = (size_t)hdr[0], t = (size_t)hdr[1], nd = (size_t)hdr[2], lo = (size_t)hdr[3], hi = (size_t)hdr[4];
    const size_t m = nd * (hi - lo);
    uint8_t* commits = slurp(f, 32 * nd * t);
    uint8_t* shares = slurp(f, 32 * m);
    uint8_t* want = slurp(f, m);
    fclose(f);
    uint8_t* v = malloc(m);
    kb_ctx* ctx = NULL;
    if (kb_ctx_create(0, &ctx) != KB_OK) return 3;
    int fails = 0;
    size_t mismatches = 0;
    for (int mode = KB_ROUND_CHECK_EXACT; mode <= KB_ROUND_CHECK_BATCHED; mode++) {
        uint64_t fb = 99;
        if (kb_ctx_set_round_check(ctx, mode) != KB_OK) fails++;
        if (kb_dkg_verify_columns(ctx, n, t, 0, nd, lo, hi, KB_POINT_ENC32, commits, shares, v) != KB_OK) {
            fprintf(stderr, "kb_dkg_verify_columns: %s\n", kb_last_error(ctx));
            fails++;
            continue;
        }
        for (size_t k = 0; k < m; k++) mismatches += v[k] != want[k];
        if (kb_ctx_round_fallbacks(ctx, &fb) != KB_OK || fb != 0) fails++;
    }
    if (kb_dkg_verify_columns(ctx, n, t, 0, nd, lo, lo, KB_POINT_ENC32, commits, shares, v) != KB_ERR_ARG) fails++;
    if (kb_dkg_verify_columns(ctx, n, t, 0, nd, lo, n + 1, KB_POINT_ENC32, commits, shares, v) != KB_ERR_ARG) fails++;
    if (kb_dkg_verify_columns(ctx, n, t, 1, 0, lo, hi, KB_POINT_ENC32, commits, shares, v) != KB_ERR_ARG) fails++;
    if (kb_dkg_verify_columns(ctx, n, t, 0, nd, lo, hi, 2, commits, shares, v) != KB_ERR_ARG) fails++;
    if (kb_dkg_verify_columns(ctx, n, t, nd, nd, lo, hi, KB_POINT_ENC32, commits, shares, v) != KB_OK) fails++;
    kb_ctx_destroy(ctx);
    printf("mismatches=%zu fails=%d\n", mismatches, fails);
    free(commits);
    free(shares);
    free(want);
    free(v);
    return (mismatches == 0 && fails == 0) ? 0 : 1;
}
