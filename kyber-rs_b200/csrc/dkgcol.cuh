// dkgcol.cuh — the share checks of a DKG round for a range of verifiers (kb_dkg_verify_columns, DESIGN §3.11): column i is
// what participant i runs in process_deal (dkg.rs:513-597), the n dealers' polynomials evaluated at the same x = i + 1.
//
// The whole curve group has exponent 8L, so for every commitment C (torsion included) x^j C = e_j C with e_j = x^j mod 8L,
// and the evaluation that PubPoly::eval computes with the exact integer x is
//     eval_d(x) = sum_j e_j C_(d,j)
// exactly.  The e_j are shared by every dealer of the column: that is the shared-scalar multi-scalar multiplication of
// dkgrlc.cuh (k_rc_sort, kb_rc_chunk, kb_rc_fold) with the weights w_j replaced by the e_j of each column, and one window
// more, since 8L > 2^255.  No randomness and no fallback: the verdict of a (column, dealer) is eval_d(x) == s B, compared as
// k_poly_eval compares, with the same base multiplication on the raw share bytes.
#pragma once
#include "dkgrlc.cuh"

#define KB_COL_WINDOWS 33   // signed radix-256 digits of an exponent < 8L < 2^255 + 2^128: window 32 is the final carry

// e = the integer in [0, 8L) that is a mod L and r8 mod 8 (a < L).  L = 5 mod 8 and 5 * 5 = 1 mod 8, so e = a + k L with
// k = 5 (r8 - a) mod 8.
KB_FN void kb_col_exponent(uint32_t* e, const uint32_t* a, uint32_t r8)
{
    const uint32_t l[8] = KB_L_WORDS;
    const uint64_t k = ((r8 - a[0]) * 5u) & 7u;
    uint64_t carry = 0;
    KB_UNROLL
    for (int w = 0; w < 8; w++) {
        const uint64_t v = (uint64_t)a[w] + k * l[w] + carry;
        e[w] = (uint32_t)v;
        carry = v >> 32;
    }
}
// signed radix-256 digits of e < 8L: e[k] in [-127, 128], e = sum_k e[k] 256^k.  Byte 31 of e is at most 0x80, so digit 31
// is negative exactly when it carries out, and that carry is digit 32.
KB_FN void kb_col_recode(int16_t* dig, const uint32_t* e)
{
    kb_rc_recode256(dig, e);
    dig[KB_COL_WINDOWS - 1] = dig[KB_RC_WINDOWS - 1] < 0 ? 1 : 0;
}
// a = x^j mod L, r8 = x^j mod 8
KB_FN void kb_col_power(uint32_t* a, uint32_t& r8, uint64_t x, uint64_t j)
{
    const uint32_t one[8] = {1, 0, 0, 0, 0, 0, 0, 0};
    kb_rc_pow_times(a, one, x, j);
    r8 = 1;
    KB_NOUNROLL
    for (uint64_t q = 0; q < j && r8; q++) r8 = (r8 * (uint32_t)x) & 7u;
}
// eval == sb as Point::eq sees it (canonical encodings): X1 Z2 = X2 Z1 and Y1 Z2 = Y2 Z1, Z never vanishes on the curve
KB_FN uint32_t kb_col_same(const ge_p3& v, const ge_p3& h)
{
    fe l, r, df;
    fe_mul(l, v.X, h.Z);
    fe_mul(r, h.X, v.Z);
    fe_sub(df, l, r);
    uint32_t same = fe_is_zero(df);
    fe_mul(l, v.Y, h.Z);
    fe_mul(r, h.Y, v.Z);
    fe_sub(df, l, r);
    return same & fe_is_zero(df);
}

#if !defined(KB_HOST_EMU)
// thread (column c, chunk of KB_RC_POW_J exponents): dig[(c KB_COL_WINDOWS + k) t + j] = digit k of (x0 + c)^j mod 8L
static __global__ void __launch_bounds__(KB_THREADS) k_col_digits(size_t kc, size_t t, uint64_t x0, int16_t* dig)
{
    const size_t jchunks = (t + KB_RC_POW_J - 1) / KB_RC_POW_J;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t c = idx / jchunks, j0 = (idx % jchunks) * KB_RC_POW_J;
    if (c >= kc) return;
    const uint64_t x = x0 + c;
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0}, xw[8] = {(uint32_t)x, (uint32_t)(x >> 32), 0, 0, 0, 0, 0, 0};
    uint32_t a[8], e[8], r8;
    int16_t d[KB_COL_WINDOWS];
    kb_col_power(a, r8, x, j0);
    const size_t j1 = j0 + KB_RC_POW_J < t ? j0 + KB_RC_POW_J : t;
    KB_NOUNROLL
    for (size_t j = j0; j < j1; j++) {
        kb_col_exponent(e, a, r8);
        kb_col_recode(d, e);
        KB_UNROLL
        for (int k = 0; k < KB_COL_WINDOWS; k++) dig[(c * KB_COL_WINDOWS + k) * t + j] = d[k];
        sc_muladd(a, a, xw, zero);
        r8 = (r8 * (uint32_t)x) & 7u;
    }
}
// thread (window w of all kc * KB_COL_WINDOWS, chunk q, dealer d): parts[((w nch + q) nd + d)] = the chunk's share of
// window w's bucket sum (k_rc_msm over more windows)
static __global__ void __launch_bounds__(KB_THREADS) k_col_msm(size_t nd, size_t t, size_t nwin, size_t nch, const uint32_t* dec, const uint32_t* ent, const uint8_t* bkt, const uint32_t* cnt,
                                                                uint32_t* parts)
{
    const size_t nd32 = (nd + 31) & ~(size_t)31;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t wq = idx / nd32, d = idx % nd32;
    if (wq >= nwin * nch || d >= nd) return;
    const size_t w = wq / nch, q = wq % nch, m = cnt[w];
    ge_p3 r;
    kb_rc_chunk(r, ent + w * t, bkt + w * t, m * q / nch, m * (q + 1) / nch, [&](uint32_t j, ge_p3& P) { kb_load_p3_w128(P, KB_FD_AT(dec, j, d, nd)); });
    kb_store_p3_w128(parts + (wq * nd + d) * 32, r);
}
// thread (column c of this group, dealer d): eval_d(x) by the fold over the windows, s B for the share, the comparison.
// Shares and verdicts are [d][kc_all]; this group's columns start at c0.
static __global__ void __launch_bounds__(KB_THREADS) k_col_check(size_t nd, size_t kc, size_t kc_all, size_t c0, size_t nch, const uint32_t* parts, const uint32_t* dealer_bad,
                                                                  const uint8_t* shares, const ge_precomp* table, uint8_t* verdict)
{
    extern __shared__ uint4 smem4[];
    ge_precomp* base = reinterpret_cast<ge_precomp*>(smem4);
    kb_stage(reinterpret_cast<uint32_t*>(base), reinterpret_cast<const uint32_t*>(table), 64 * 8 * 24);
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= kc * nd) return;   // no block barrier below
    const size_t c = idx / nd, d = idx % nd, slot = d * kc_all + c0 + c;
    ge_p3 W, h;
    kb_rc_fold<KB_COL_WINDOWS>(W, nch, [&](size_t k, size_t q, ge_p3& P) { kb_load_p3_w128(P, parts + (((c * KB_COL_WINDOWS + k) * nch + q) * nd + d) * 32); });
    uint32_t s[8];
    int8_t e[64];
    kb_load32(s, shares, slot);
    sc_recode16(e, s);
    ge_scalarmult_base<true>(h, e, base);
    verdict[slot] = (uint8_t)(kb_col_same(W, h) & (dealer_bad[d] ? 0u : 1u));
}
// the items of the per-share path: item k = (dealer k / kc, verifier ver_lo + k % kc), the layout of the verdicts
static __global__ void __launch_bounds__(KB_THREADS) k_col_items(size_t m, size_t kc, size_t ver_lo, uint32_t* poly_id, uint32_t* idx)
{
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    poly_id[k] = (uint32_t)(k / kc);
    idx[k] = (uint32_t)(ver_lo + k % kc);
}
#endif  // !KB_HOST_EMU
