// ops.cuh — per-thread algorithms: table selection, scalar multiplication, byte-level point
// checks and the EdDSA / Schnorr verification state machine.  One GPU thread owns one item
// (scalar, point, signature); the kernels in kernels.cu are thin launch wrappers around these.
//
// Citations are to /root/reference/src.
#pragma once
#include "fe.cuh"
#include "ge.cuh"
#include "sc.cuh"
#include "sha512.cuh"
#include "half.cuh"

// kb_sig_status (include/kyber_b200.h) — sign/error.rs:6-25
#define KB_SIG_OK 0
#define KB_SIG_LENGTH 1
#define KB_SIG_NOT_CANONICAL 2
#define KB_SIG_R_NOT_CANONICAL 3
#define KB_SIG_R_SMALL_ORDER 4
#define KB_SIG_PK_NOT_CANONICAL 5
#define KB_SIG_PK_SMALL_ORDER 6
#define KB_SIG_MARSHALLING 7
#define KB_SIG_INVALID 8

// ---------------------------------------------------------------------------------------
// byte-level checks on a 32-byte encoding held as 8 little-endian words
// ---------------------------------------------------------------------------------------
// Point::is_canonical (group/edwards25519/point.rs:322-337), bug-compatible: the low-byte
// test is 0xED - (1 - b[0]) in wrapping u16, so with bytes 1..30 = 0xff and b[31]&0x7f = 0x7f
// the encoding is reported NON-canonical for every b[0] >= 0x14 (SURVEY §A1).
KB_FN uint32_t pt_is_canonical(const uint32_t* w)
{
    uint32_t ones = ((w[7] & 0x7fffffffu) == 0x7fffffffu) & ((w[0] >> 8) == 0x00ffffffu);
    KB_UNROLL
    for (int i = 1; i < 7; i++) ones &= (w[i] == 0xffffffffu);
    return !(ones & ((w[0] & 0xffu) >= 0x14u));
}
// Point::has_small_order (point.rs:286-310) for an encoding that is canonical and on the
// curve: the reference re-encodes the decoded point and compares bytes 0..30 and byte 31
// & 0x7f with WEAK_KEYS (constants.rs:3744); for such encodings the re-encoding equals the
// input up to bit 255, so the comparison can run on the raw words.
KB_FN uint32_t pt_is_small_order_bytes(const uint32_t* w)
{
    const uint32_t top = w[7] & 0x7fffffffu;
    uint32_t mid0 = 1, midf = 1;
    KB_UNROLL
    for (int i = 1; i < 7; i++) {
        mid0 &= (w[i] == 0u);
        midf &= (w[i] == 0xffffffffu);
    }
    uint32_t k0 = mid0 & (top == 0u) & (w[0] == 0u);                 // y = 0      (order 4)
    uint32_t k1 = mid0 & (top == 0u) & (w[0] == 1u);                 // y = 1      (order 1)
    uint32_t k4 = midf & (top == 0x7fffffffu) & (w[0] == 0xffffffecu);  // y = p - 1  (order 2)
    const uint32_t o8a[8] = {0x8f95e826u, 0xb027b2c2u, 0x89f4c345u, 0xf098eff2u, 0x05acdfd5u, 0x3933c6d3u, 0x880238b1u, 0x05fc536du};
    const uint32_t o8b[8] = {0x706a17c7u, 0x4fd84d3du, 0x760b3cbau, 0x0f67100du, 0xfa53202au, 0xc6cc392cu, 0x77fdc74eu, 0x7a03ac92u};
    uint32_t k2 = (top == o8a[7]), k3 = (top == o8b[7]);
    KB_UNROLL
    for (int i = 0; i < 7; i++) {
        k2 &= (w[i] == o8a[i]);
        k3 &= (w[i] == o8b[i]);
    }
    return k0 | k1 | k2 | k3 | k4;
}

// ---------------------------------------------------------------------------------------
// table selection
// ---------------------------------------------------------------------------------------
// select_cached (ge.rs:488-500): c = d * P from tbl[j] = (j+1) P, d in [-8, 8]; d = 0 gives
// the identity.  CT=true scans all 8 entries with conditional moves (no secret-dependent
// address or branch); CT=false indexes directly (public scalars only).
template <bool CT>
KB_FN void ge_select_cached(ge_cached& c, const ge_cached* tbl, int d)
{
    const uint32_t neg = (uint32_t)d >> 31;
    const int babs = (d ^ -(int)neg) + (int)neg;
    ge_cached_identity(c);
    if (CT) {
        KB_NOUNROLL
        for (int j = 0; j < 8; j++) {
            const uint32_t hit = (uint32_t)(babs == j + 1);
            fe_cmov(c.YpX, tbl[j].YpX, hit);
            fe_cmov(c.YmX, tbl[j].YmX, hit);
            fe_cmov(c.T2d, tbl[j].T2d, hit);
            fe_cmov(c.Z, tbl[j].Z, hit);
        }
    } else {
        if (babs != 0) c = tbl[babs - 1];
    }
    ge_cached_cneg(c, neg);
}
// select_pre_computed (ge.rs:423-434) on one window of the base-point table
template <bool CT>
KB_FN void ge_select_precomp(ge_precomp& c, const ge_precomp* win, int d)
{
    const uint32_t neg = (uint32_t)d >> 31;
    const int babs = (d ^ -(int)neg) + (int)neg;
    ge_precomp_identity(c);
    if (CT) {
        KB_NOUNROLL
        for (int j = 0; j < 8; j++) {
            const uint32_t hit = (uint32_t)(babs == j + 1);
            fe_cmov(c.ypx, win[j].ypx, hit);
            fe_cmov(c.ymx, win[j].ymx, hit);
            fe_cmov(c.xy2d, win[j].xy2d, hit);
        }
    } else {
        if (babs != 0) c = win[babs - 1];
    }
    ge_precomp_cneg(c, neg);
}

// tbl[j] = (j+1) P, j = 0..7   (ge.rs:537-543)
KB_FN void ge_build_table8(ge_cached* tbl, const ge_p3& p)
{
    ge_p3 m = p;
    ge_to_cached(tbl[0], p);
    KB_NOUNROLL
    for (int j = 1; j < 8; j++) {
        ge_add<true>(m, m, tbl[0]);
        ge_to_cached(tbl[j], m);
    }
}

// ---------------------------------------------------------------------------------------
// scalar multiplication
// ---------------------------------------------------------------------------------------
// KB_LOCKSTEP(): a block barrier at the top of every window iteration of the long scalar-multiplication
// loops.  It is not needed for correctness — it keeps the warps of a block on the same instructions, which
// is what the instruction cache wants (the loop body is tens of KB; warps drifting apart showed up in ncu as
// `no_instruction` stalls, icc hit rate 85 %).  Measured on verify: 35.4 -> 38.3 M signatures/s.  Callers
// must therefore keep EVERY thread of the block inside the loop (tail threads redo the last item and skip
// the store; items off the fast path multiply the identity).
#if defined(KB_HOST_EMU)
#define KB_LOCKSTEP()
#else
#define KB_LOCKSTEP() __syncthreads()
#endif
// h = a * P, ge_scalar_mult (ge.rs:508-568): signed radix-16 fixed window over the
// per-thread table tbl[8]; e = sc_recode16(a).  LOCKSTEP = false drops the block barrier, for callers
// that run it in a divergent branch (k_keyset_mul).
template <bool CT, bool LOCKSTEP = true>
KB_FN void ge_scalarmult(ge_p3& h, const int8_t* e, const ge_cached* tbl)
{
    ge_cached c;
    ge_identity(h);
    // one doubling body and one addition body in the loop (runtime T flags): keeps the loop small
    // enough for the instruction cache
    KB_NOUNROLL
    for (int i = 63; i >= 0; i--) {
        if (LOCKSTEP) { KB_LOCKSTEP(); }
        if (i != 63) {
            KB_NOUNROLL
            for (int k = 0; k < 4; k++) ge_dbl_rt(h, h, k == 3);
        }
        ge_select_cached<CT>(c, tbl, e[i]);
        ge_add_rt(h, h, c, i == 0);
    }
}
// h = a * B, ge_scalar_mult_base (ge.rs:442-486) restated as a 64-window comb:
// base[w*8 + j] = (j+1) * 16^w * B, so no doublings are needed at all.
template <bool CT>
KB_FN void ge_scalarmult_base(ge_p3& h, const int8_t* e, const ge_precomp* base, int w_lo = 0, int w_hi = 64)
{
    ge_precomp c;
    ge_identity(h);
    KB_NOUNROLL
    for (int w = w_lo; w < w_hi; w++) {
        ge_select_precomp<CT>(c, base + 8 * w, e[w]);
        ge_madd<true>(h, h, c);
    }
}
// signed radix-256 digits of a scalar < 2^253: d[0..31] in (-128, 128]
KB_FN void sc_recode256(int16_t* d, const uint32_t* s)
{
    int carry = 0;
    KB_UNROLL
    for (int i = 0; i < 32; i++) {
        int v = (int)((s[i >> 2] >> (8 * (i & 3))) & 255u) + carry;
        carry = v > 128;
        d[i] = (int16_t)(v - (carry << 8));
    }
}
// h = s * B + k * A (public data), Straus with shared doublings; the fixed base uses signed
// radix-256 digits against base128[j] = (j+1) B, j = 0..127 (one mixed addition every EIGHT
// doublings instead of every four), the variable base signed radix-16 digits against the
// per-thread table tbl[j] = (j+1) A.
KB_FN void ge_double_scalarmult_vartime(ge_p3& h, const int16_t* ds, const int8_t* ek, const ge_cached* tbl, const ge_precomp* base128)
{
    ge_cached c;
    ge_identity(h);
    KB_NOUNROLL
    for (int i = 63; i >= 0; i--) {
        KB_LOCKSTEP();
        if (i != 63) {
            KB_NOUNROLL
            for (int k = 0; k < 4; k++) ge_dbl_rt(h, h, k == 3);
        }
        // the fixed-base entry is widened to the cached form (Z = 1) so that both additions of an even
        // step run through the SAME code (one multiplication by 1 more, ~1000 instructions less)
        const int nadd = (i & 1) ? 1 : 2;
        KB_NOUNROLL
        for (int a = 0; a < nadd; a++) {
            if (a == 0) {
                ge_select_cached<false>(c, tbl, ek[i]);
            } else {
                const int d = ds[i >> 1];
                const uint32_t neg = (uint32_t)d >> 31;
                const int babs = (d ^ -(int)neg) + (int)neg;
                ge_cached_identity(c);
                if (babs != 0) {
                    c.YpX = base128[babs - 1].ypx;
                    c.YmX = base128[babs - 1].ymx;
                    c.T2d = base128[babs - 1].xy2d;
                }
                ge_cached_cneg(c, neg);
            }
            ge_add_rt(h, h, c, (a + 1 < nadd) || i == 0);
        }
    }
}

// ---------------------------------------------------------------------------------------
// EdDSA / Schnorr verification
// ---------------------------------------------------------------------------------------
// Both verifiers check compress(s*B - h*A) == R-bytes, which is the reference's
// "R + h*A == s*B on canonical encodings" (eddsa_sig.rs:201-210, schnorr_sig.rs:96-106)
// once R is canonical, on the curve and not of small order.  When that fast path does not
// accept, the reference's own check ORDER decides which error is reported; deciding it
// needs to know whether R decodes, which is only computed then.
//
// SCHNORR=false: eddsa::verify_with_checks (sign/eddsa/eddsa_sig.rs:159-212)
// SCHNORR=true : schnorr::verify_with_checks (sign/schnorr/schnorr_sig.rs:53-110); its
//   challenge hashes the re-encoded R and A (:128-141), which equal the raw bytes whenever
//   the fast path is entered.
//
// The work is split so that the final compression can share one field inversion between
// several signatures (Montgomery's trick, kernels.cuh):
//   sig_stage1   byte-level checks, decompress A, challenge hash, Q = s*B - h*A  -> flags, Q
//   sig_finish   compare compress(Q) with the R bytes / classify the failure      -> status
#define KB_F_SC 1u     // s canonical           (scalar.rs:54)
#define KB_F_RC 2u     // R canonical           (point.rs:322)
#define KB_F_RS 4u     // R small order         (point.rs:286)
#define KB_F_AC 8u     // A canonical
#define KB_F_AS 16u    // A small order
#define KB_F_AOK 32u   // A decodes             (ge.rs:124)
#define KB_F_FAST 64u  // Q was computed

template <bool SCHNORR>
KB_FN uint32_t sig_stage1(ge_p3& Q, const uint32_t* pk_w, const uint32_t* sig_w, const uint8_t* msg, uint64_t mlen, const ge_precomp* base128, ge_cached* tbl)
{
    const uint32_t* r_w = sig_w;
    const uint32_t* s_w = sig_w + 8;
    uint32_t f = 0;
    f |= sc_is_canonical(s_w) ? KB_F_SC : 0u;
    f |= pt_is_canonical(r_w) ? KB_F_RC : 0u;
    f |= pt_is_small_order_bytes(r_w) ? KB_F_RS : 0u;
    f |= pt_is_canonical(pk_w) ? KB_F_AC : 0u;
    f |= pt_is_small_order_bytes(pk_w) ? KB_F_AS : 0u;
    ge_identity(Q);
    // EdDSA never looks at A when an earlier check fails; Schnorr decodes A before is_canonical(A)
    const uint32_t pre_ok = (f & (KB_F_SC | KB_F_RC | KB_F_RS)) == (KB_F_SC | KB_F_RC);
    // Every thread of the block runs the whole scalar multiplication (its loop holds a block barrier, see
    // KB_LOCKSTEP); items that are not on the fast path run it on the identity and drop the result.
    ge_p3 A;
    const uint32_t a_dec = ge_decompress(A, pk_w);
    if (SCHNORR || (pre_ok && (f & KB_F_AC))) f |= a_dec ? KB_F_AOK : 0u;
    const bool fast = pre_ok && (f & (KB_F_AC | KB_F_AS | KB_F_AOK)) == (KB_F_AC | KB_F_AOK);
    int16_t ds[32];
    int8_t ek[64];
    ge_p3 nA;
    if (fast) {
        uint32_t digest[16], hk[8];
        sha512_ram(digest, r_w, pk_w, msg, mlen);
        sc_reduce512(hk, digest);
        sc_recode256(ds, s_w);
        sc_recode16(ek, hk);
        ge_neg(nA, A);
    } else {
        for (int i = 0; i < 32; i++) ds[i] = 0;
        for (int i = 0; i < 64; i++) ek[i] = 0;
        ge_identity(nA);
    }
    ge_build_table8(tbl, nA);
    ge_double_scalarmult_vartime(Q, ds, ek, tbl, base128);
    if (!fast) {
        ge_identity(Q);
        return f;
    }
    return f | KB_F_FAST;
}
// The first failing check in the reference's order (the signature is known not to verify).  r_ok = "R decodes"
// (ge.rs:124) is only looked at where the reference would have reached the decode.
template <bool SCHNORR>
KB_FN uint32_t sig_classify(uint32_t f, uint32_t r_ok)
{
    if (!SCHNORR) {
        if (!(f & KB_F_SC)) return KB_SIG_NOT_CANONICAL;
        if (!(f & KB_F_RC)) return KB_SIG_R_NOT_CANONICAL;
        if (f & KB_F_RS) return KB_SIG_R_SMALL_ORDER;  // weak encodings are on the curve
    }
    if (!r_ok) return KB_SIG_MARSHALLING;
    if (SCHNORR) {
        if (!(f & KB_F_RC)) return KB_SIG_R_NOT_CANONICAL;
        if (f & KB_F_RS) return KB_SIG_R_SMALL_ORDER;
        if (!(f & KB_F_SC)) return KB_SIG_NOT_CANONICAL;
        if (!(f & KB_F_AOK)) return KB_SIG_MARSHALLING;
        if (!(f & KB_F_AC)) return KB_SIG_PK_NOT_CANONICAL;
    } else {
        if (!(f & KB_F_AC)) return KB_SIG_PK_NOT_CANONICAL;
        if (!(f & KB_F_AOK)) return KB_SIG_MARSHALLING;
    }
    if (f & KB_F_AS) return KB_SIG_PK_SMALL_ORDER;
    return KB_SIG_INVALID;
}
// enc = compress(Q) (only meaningful with KB_F_FAST)
template <bool SCHNORR>
KB_FN uint32_t sig_finish(uint32_t f, const uint32_t* enc, const uint32_t* r_w)
{
    if (f & KB_F_FAST) {
        uint32_t diff = 0;
        KB_UNROLL
        for (int i = 0; i < 8; i++) diff |= enc[i] ^ r_w[i];
        if (diff == 0) return KB_SIG_OK;
    }
    uint32_t r_ok = 1;
    const bool r_reached = SCHNORR || (f & (KB_F_SC | KB_F_RC | KB_F_RS)) == (KB_F_SC | KB_F_RC);
    if (r_reached && !(f & KB_F_RS)) {
        ge_p3 R;
        r_ok = ge_decompress(R, r_w);
    }
    return sig_classify<SCHNORR>(f, r_ok);
}
// one signature start to finish (own inversion) — the composition the two-stage kernels implement
template <bool SCHNORR>
KB_FN uint32_t sig_verify(const uint32_t* pk_w, const uint32_t* sig_w, const uint8_t* msg, uint64_t mlen, const ge_precomp* base128, ge_cached* tbl)
{
    ge_p3 Q;
    const uint32_t f = sig_stage1<SCHNORR>(Q, pk_w, sig_w, msg, mlen, base128, tbl);
    uint32_t enc[8];
    ge_compress(enc, Q);
    return sig_finish<SCHNORR>(f, enc, sig_w);
}

// ---------------------------------------------------------------------------------------
// the same verifiers with half-size scalars (half.cuh): 128 doublings instead of 253
// ---------------------------------------------------------------------------------------
//   W = (u*s mod L)*B + |v|*A' + u*R',   A' = -sign(v)*A,  R' = -R,   accept <=> W is the identity
// with (u, v) = sc_half(h).  One signed radix-16 table each for A' and R' (tbl[0..7], tbl[8..15]) inside the
// doubling loop.  The multiple of B needs no doublings at all: it is a comb over a table that is computed once
// per context and shared by every signature, comb[p][j] = (j+1) * 2^(17 p) * B, p = 0..14, j = 0..65535 (94 MB;
// the first version had 13-bit windows: 20 positions, 7.9 MB): 15 additions after the loop instead of 32 inside it.  The number of windows is BLOCK-uniform
// (the loop holds a block barrier): the kernel takes the maximum over its threads, 33 for almost every block
// of honest input.
#define KB_F_ROK 128u  // R decodes            (ge.rs:124)
#define KB_HALF_MIN_WINDOWS 1
// Window width of the comb.  Every position less is one addition less per signature (0.08 ms per 2^20 signatures); the
// operands are fetched one step ahead, so it does not matter that a wider table no longer fits the L2.  Measured on one
// B200 (profiles/r2_ab_comb*.txt), k_verify_half_main for 2^20 signatures: 13 bits x 20 positions (7.9 MB) 16.35 ms,
// 14 x 19 16.28, 15 x 17 (27 MB) 16.10, 16 x 16 (50 MB) 16.03, 17 x 15 (94 MB) 15.95.  19 x 14 would take 352 MB for one more.
#ifndef KB_HALF_JOINT
#define KB_HALF_JOINT 1   // one joint radix-4 table for A' and R' instead of two radix-16 tables (below)
#endif
#ifndef KB_COMB_BITS
#define KB_COMB_BITS 17
#define KB_COMB_POS 15
#endif
static_assert(KB_COMB_BITS * KB_COMB_POS >= 254 && KB_COMB_BITS <= 20, "the comb must cover 253 bits and the recoding carry");
#define KB_COMB_HALF (1 << (KB_COMB_BITS - 1))
#if KB_COMB_BITS > 15
typedef int32_t kb_comb_digit;
#else
typedef int16_t kb_comb_digit;
#endif

// signed radix-2^KB_COMB_BITS digits of a scalar < 2^253: d[0..KB_COMB_POS) in (-KB_COMB_HALF, KB_COMB_HALF]
KB_FN void sc_recode_comb(kb_comb_digit* d, const uint32_t* s)
{
    int carry = 0;
    KB_UNROLL
    for (int p = 0; p < KB_COMB_POS; p++) {
        const int bit = KB_COMB_BITS * p, wi = bit >> 5, sh = bit & 31;
        uint32_t x = s[wi] >> sh;
        if (sh + KB_COMB_BITS > 32 && wi + 1 < 8) x |= s[wi + 1] << (32 - sh);
        int v = (int)(x & ((1u << KB_COMB_BITS) - 1u)) + carry;
        carry = v > KB_COMB_HALF;
        d[p] = (kb_comb_digit)(v - (carry << KB_COMB_BITS));
    }
}
KB_FN void kb_ld_precomp(ge_cached& c, const ge_precomp* e)
{
#if defined(KB_HOST_EMU)
    c.YpX = e->ypx;
    c.YmX = e->ymx;
    c.T2d = e->xy2d;
#else
    const uint4* q = reinterpret_cast<const uint4*>(e);
    uint4 a;
    a = __ldg(q + 0); c.YpX.v[0] = a.x; c.YpX.v[1] = a.y; c.YpX.v[2] = a.z; c.YpX.v[3] = a.w;
    a = __ldg(q + 1); c.YpX.v[4] = a.x; c.YpX.v[5] = a.y; c.YpX.v[6] = a.z; c.YpX.v[7] = a.w;
    a = __ldg(q + 2); c.YmX.v[0] = a.x; c.YmX.v[1] = a.y; c.YmX.v[2] = a.z; c.YmX.v[3] = a.w;
    a = __ldg(q + 3); c.YmX.v[4] = a.x; c.YmX.v[5] = a.y; c.YmX.v[6] = a.z; c.YmX.v[7] = a.w;
    a = __ldg(q + 4); c.T2d.v[0] = a.x; c.T2d.v[1] = a.y; c.T2d.v[2] = a.z; c.T2d.v[3] = a.w;
    a = __ldg(q + 5); c.T2d.v[4] = a.x; c.T2d.v[5] = a.y; c.T2d.v[6] = a.z; c.T2d.v[7] = a.w;
#endif
}

// What the preparation hands to the main loop: the two operand points (affine, Z = 1), the three scalars.
struct kb_half_rec {
    fe ax, ay, at;    // A' = -sign(v) * A
    fe rx, ry, rt;    // R' = -R
    uint32_t w[8];    // u*s mod L
    uint32_t u[8];    // odd, > 0
    uint32_t v[8];    // |v|
    uint32_t f;       // KB_F_* flags
    int nwin;         // windows this signature needs (0 when it is off the fast path)
};
// The preparation is two independent phases — the kernel runs them in either order (kernels.cuh):
//   points   decompress A and R (multiplier-bound)          -> -A, -R and the two "decodes" bits
//   scalars  byte-level checks, challenge hash, lattice step, u*s mod L (ALU-bound) -> w, u, |v|, sign(v), window count
// -P for the encoding w (affine X, Y, T); returns 1 if w decodes
KB_FN uint32_t sig_half_point(fe& x, fe& y, fe& t, const uint32_t* w)
{
    ge_p3 p;
    const uint32_t ok = ge_decompress(p, w);
    fe_neg(x, p.X);
    y = p.Y;
    fe_neg(t, p.T);
    return ok;
}
struct kb_half_sc {
    uint32_t w[8], u[8], v[8];
    uint32_t f;      // byte-level flags (KB_F_SC, RC, RS, AC, AS)
    uint32_t vneg;   // v < 0: A' = +A
    int nwin;
};
// The hash and the lattice step run for every signature that passes the byte-level checks (whether A and R decode is not
// known here; sig_half_flags decides).
template <bool SCHNORR>
KB_FN void sig_half_scalars(kb_half_sc& sc, const uint32_t* pk_w, const uint32_t* sig_w, const uint8_t* msg, uint64_t mlen)
{
    const uint32_t* r_w = sig_w;
    const uint32_t* s_w = sig_w + 8;
    uint32_t f = 0;
    f |= sc_is_canonical(s_w) ? KB_F_SC : 0u;
    f |= pt_is_canonical(r_w) ? KB_F_RC : 0u;
    f |= pt_is_small_order_bytes(r_w) ? KB_F_RS : 0u;
    f |= pt_is_canonical(pk_w) ? KB_F_AC : 0u;
    f |= pt_is_small_order_bytes(pk_w) ? KB_F_AS : 0u;
    sc.f = f;
    sc.vneg = 0;
    sc.nwin = 0;
    if ((f & (KB_F_SC | KB_F_RC | KB_F_RS | KB_F_AC | KB_F_AS)) == (KB_F_SC | KB_F_RC | KB_F_AC)) {
        uint32_t digest[16], hk[8];
        const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        sha512_ram(digest, r_w, pk_w, msg, mlen);
        sc_reduce512(hk, digest);
        kb_halfsc hs;
        sc_half(hs, hk);
        sc_muladd(sc.w, hs.u, s_w, zero);
        KB_UNROLL
        for (int i = 0; i < 8; i++) {
            sc.u[i] = hs.u[i];
            sc.v[i] = hs.v[i];
        }
        sc.vneg = hs.vneg;
        sc.nwin = hs.bits / 4 + 1;
    } else {
        KB_UNROLL
        for (int i = 0; i < 8; i++) sc.w[i] = sc.u[i] = sc.v[i] = 0;
    }
}
// byte-level flags + the "decodes" bits (bit 0: A, bit 1: R) -> the flags the main loop and sig_classify read
template <bool SCHNORR>
KB_FN uint32_t sig_half_flags(uint32_t f, uint32_t dec)
{
    const uint32_t pre_ok = (f & (KB_F_SC | KB_F_RC | KB_F_RS)) == (KB_F_SC | KB_F_RC);
    f |= (dec & 2u) ? KB_F_ROK : 0u;
    // EdDSA never looks at A when an earlier check fails; Schnorr decodes A before is_canonical(A)
    if (SCHNORR || (pre_ok && (f & KB_F_AC))) f |= (dec & 1u) ? KB_F_AOK : 0u;
    const bool fast = pre_ok && (dec & 2u) && (f & (KB_F_AC | KB_F_AS | KB_F_AOK)) == (KB_F_AC | KB_F_AOK);
    return fast ? (f | KB_F_FAST) : f;
}
// what a signature off the fast path hands to the main loop: neutral operands, no windows
KB_FN void sig_half_rec_neutral(kb_half_rec& rec)
{
    KB_UNROLL
    for (int i = 0; i < 8; i++) rec.w[i] = rec.u[i] = rec.v[i] = 0;
    fe_set(rec.ax, 0); fe_set(rec.ay, 1); fe_set(rec.at, 0);
    fe_set(rec.rx, 0); fe_set(rec.ry, 1); fe_set(rec.rt, 0);
    rec.nwin = 0;
}
// A' = -sign(v) * A from -A
KB_FN void sig_half_apply_vneg(fe& ax, fe& at, uint32_t vneg)
{
    fe nx, nt;
    fe_neg(nx, ax);
    fe_neg(nt, at);
    fe_cmov(ax, nx, vneg);
    fe_cmov(at, nt, vneg);
}
// both phases and the flags: the record of one signature
template <bool SCHNORR>
KB_FN void sig_half_prep(kb_half_rec& rec, const uint32_t* pk_w, const uint32_t* sig_w, const uint8_t* msg, uint64_t mlen)
{
    uint32_t dec = sig_half_point(rec.ax, rec.ay, rec.at, pk_w);
    dec |= sig_half_point(rec.rx, rec.ry, rec.rt, sig_w) << 1;
    kb_half_sc sc;
    sig_half_scalars<SCHNORR>(sc, pk_w, sig_w, msg, mlen);
    rec.f = sig_half_flags<SCHNORR>(sc.f, dec);
    if (rec.f & KB_F_FAST) {
        KB_UNROLL
        for (int i = 0; i < 8; i++) {
            rec.w[i] = sc.w[i];
            rec.u[i] = sc.u[i];
            rec.v[i] = sc.v[i];
        }
        sig_half_apply_vneg(rec.ax, rec.at, sc.vneg);
        rec.nwin = sc.nwin;
    } else {
        sig_half_rec_neutral(rec);
    }
}
// digit strings and the two per-signature tables: tbl[0..7] = 1..8 A', tbl[8..15] = 1..8 R'
KB_FN void sig_half_setup(kb_comb_digit* dw, int8_t* eu, int8_t* ev, ge_cached* tbl, const kb_half_rec& rec)
{
    sc_recode_comb(dw, rec.w);
    sc_recode16(eu, rec.u);
    sc_recode16(ev, rec.v);
    // A magnitude below 2^(4k - 1) fits k signed radix-16 digits if the top one may be +8 (the tables hold
    // 1P..8P): the standard recoding turns a top digit of 8 into (-8, carry 1); undo exactly that.
    const int k = rec.nwin;
    if (k > 0 && k < 64) {
        if (eu[k] == 1) { eu[k] = 0; eu[k - 1] = 8; }
        if (ev[k] == 1) { ev[k] = 0; ev[k - 1] = 8; }
    }
    KB_NOUNROLL
    for (int q = 0; q < 2; q++) {
        ge_p3 p;
        p.X = q ? rec.rx : rec.ax;
        p.Y = q ? rec.ry : rec.ay;
        p.T = q ? rec.rt : rec.at;
        fe_set(p.Z, 1);
        ge_build_table8(tbl + 8 * q, p);
    }
}
// W = |v|*A' + u*R' by `nwin` shared windows of four doublings, then the comb for the multiple of B.  Every thread
// of the block runs the same trip count; one addition body serves all three operands (the comb entries are widened
// to the cached form, Z = 1).
KB_FN void ge_triple_scalarmult_vartime(ge_p3& h, int nwin, const kb_comb_digit* dw, const int8_t* eu, const int8_t* ev, const ge_cached* tbl, const ge_precomp* comb)
{
    ge_identity(h);
    KB_NOUNROLL
    for (int i = nwin - 1; i >= -KB_COMB_POS; i--) {
        KB_LOCKSTEP();
        // a window = up to four doublings, then its additions; every step ends in the same four products
        const int ndbl = (i >= 0 && i != nwin - 1) ? 4 : 0;
        const int nstep = ndbl + (i >= 0 ? 2 : 1);
        KB_NOUNROLL
        for (int step = 0; step < nstep; step++) {
            fe e, f, g, hh;
            bool with_t;
            if (step < ndbl) {
                ge_dbl_front(e, f, g, hh, h);
                with_t = step == ndbl - 1;
            } else {
                const int a = step - ndbl;
                ge_cached c;
                if (i >= 0) {
                    ge_select_cached<false>(c, tbl + 8 * a, a ? eu[i] : ev[i]);
                } else {
                    const int p = -1 - i;
                    const int d = dw[p];
                    const uint32_t neg = (uint32_t)d >> 31;
                    const int babs = (d ^ -(int)neg) + (int)neg;
                    ge_cached_identity(c);
                    if (babs != 0) kb_ld_precomp(c, comb + (size_t)p * KB_COMB_HALF + (babs - 1));
                    ge_cached_cneg(c, neg);
                }
                ge_add_front(e, f, g, hh, h, c);
                // T is dead when a doubling (or the end) follows
                with_t = !((i > 0 && step + 1 == nstep) || i == -KB_COMB_POS);
            }
            ge_tail(h, e, f, g, hh, with_t);
        }
    }
}
// The same loop with the operand of every addition FETCHED ONE STEP AHEAD.  The per-thread tables live in local memory
// (2 KB per thread: L1 holds a fraction of an SM's 768 KB, most entries come from L2), and in the loop above an addition
// starts with two dependent loads (digit -> table entry) right in front of its first multiplication: ncu's source view
// (round 2) charges 7 % of the kernel's stall samples to exactly those loads (long scoreboard).  Here the raw entry of
// the NEXT addition is requested between the front end and the four closing products of the CURRENT step (about 800
// instructions of cover); only the identity / negation selects wait for it, at the point of use.  While the closing
// products run, 32 more registers are live than before — they fit under the kernel's 168.
struct kb_operand {
    ge_cached c;     // raw table / comb entry (for comb entries c.Z is not loaded)
    uint32_t neg;    // negate it
    uint32_t nz;     // digit != 0 (otherwise the operand is the identity and c is ignored)
};
// operand of addition `a` (0: A' with ev, 1: R' with eu) of window i >= 0, or of comb position -1 - i for i < 0
KB_FN void kb_operand_fetch(kb_operand& o, int i, int a, const kb_comb_digit* dw, const int8_t* eu, const int8_t* ev, const ge_cached* tbl, const ge_precomp* comb)
{
    int d;
    if (i >= 0) d = a ? eu[i] : ev[i];
    else d = dw[-1 - i];
    o.neg = (uint32_t)d >> 31;
    const int babs = (d ^ -(int)o.neg) + (int)o.neg;
    o.nz = (uint32_t)(babs != 0);
    const int idx = babs != 0 ? babs - 1 : 0;   // always a valid entry: the loads are unconditional
    if (i >= 0) o.c = tbl[8 * a + idx];
    else kb_ld_precomp(o.c, comb + (size_t)(-1 - i) * KB_COMB_HALF + idx);
}
KB_FN void kb_operand_use(ge_cached& c, const kb_operand& o, bool is_comb)
{
    ge_cached id;
    ge_cached_identity(id);
    c = o.c;
    if (is_comb) fe_set(c.Z, 1);
    fe_cmov(c.YpX, id.YpX, o.nz ^ 1u);
    fe_cmov(c.YmX, id.YmX, o.nz ^ 1u);
    fe_cmov(c.T2d, id.T2d, o.nz ^ 1u);
    fe_cmov(c.Z, id.Z, o.nz ^ 1u);
    ge_cached_cneg(c, o.neg);
}
KB_FN void ge_triple_scalarmult_prefetch(ge_p3& h, int nwin, const kb_comb_digit* dw, const int8_t* eu, const int8_t* ev, const ge_cached* tbl, const ge_precomp* comb)
{
    ge_identity(h);
    kb_operand nx;
    kb_operand_fetch(nx, nwin - 1, 0, dw, eu, ev, tbl, comb);   // the first window has no doublings in front of it
    KB_NOUNROLL
    for (int i = nwin - 1; i >= -KB_COMB_POS; i--) {
        KB_LOCKSTEP();
        const int ndbl = (i >= 0 && i != nwin - 1) ? 4 : 0;
        const int nstep = ndbl + (i >= 0 ? 2 : 1);
        KB_NOUNROLL
        for (int step = 0; step < nstep; step++) {
            fe e, f, g, hh;
            bool with_t;
            if (step < ndbl) {
                ge_dbl_front(e, f, g, hh, h);
                with_t = step == ndbl - 1;
                if (with_t) kb_operand_fetch(nx, i, 0, dw, eu, ev, tbl, comb);   // the window's first addition follows
            } else {
                const int a = step - ndbl;
                ge_cached c;
                kb_operand_use(c, nx, i < 0);
                ge_add_front(e, f, g, hh, h, c);
                // T is dead when a doubling (or the end) follows
                with_t = !((i > 0 && step + 1 == nstep) || i == -KB_COMB_POS);
                // the next addition, unless doublings come first (then their last one fetches) or this is the end
                if (i >= 0 && a == 0) kb_operand_fetch(nx, i, 1, dw, eu, ev, tbl, comb);
                else if (i <= 0 && i > -KB_COMB_POS) kb_operand_fetch(nx, i - 1, 0, dw, eu, ev, tbl, comb);
            }
            ge_tail(h, e, f, g, hh, with_t);
        }
    }
}
// ---- JOINT windows for the two variable points (KB_HALF_JOINT, default).  Instead of one signed radix-16 table each for
// A' and R' (16 entries, two additions per four doublings) the loop uses ONE table of the combinations i R' + j A' of
// signed radix-4 digits, i in {0, 1, 2}, j in {-2 .. 2} (the sign of a digit pair is pulled out: 11 entries), and adds
// once per TWO doublings: 9 additions instead of 14 to build the tables, 65 instead of 66 additions in the loop of a
// 128-bit pair, 1.4 KB instead of 2 KB of per-thread table.  A digit pair is turned into one signed code:
// |code| - 1 = table slot, 0 = both digits zero, sign = negate the entry.
//   slot: 0 A'   1 2A'   2 R'-2A'   3 R'-A'   4 R'   5 R'+A'   6 R'+2A'   (7 unused)   8 2R'-A'   9 2R'   10 2R'+A'   11 2R'+2A'
#define KB_JOINT_SLOTS 12
// Signed radix-4 digits in [-1, 2] without a carry loop: digit_i = value_i + carry_i - 4 carry_(i+1), and a carry leaves
// digit i exactly when value_i + carry_i + 1 >= 4 — which is the carry of the plain 256-bit addition x + 0x55..55 out
// of its i-th pair of bits.  So with xk = x + 0x55..55 the digit is (pair i of xk) - 1, for every i at once.
KB_FN void sc_joint4_bias(uint32_t* xk, const uint32_t* x)
{
    const uint32_t k[8] = {0x55555555u, 0x55555555u, 0x55555555u, 0x55555555u, 0x55555555u, 0x55555555u, 0x55555555u, 0x55555555u};
    kb_add8(xk, x, k);   // x < 2^253: no carry leaves the top pair
}
// code of digit pair `idx` (0..127) of (u, v), from the biased words
KB_FN int sc_joint4_code(const uint32_t* uk, const uint32_t* vk, int idx)
{
    const int sh = 2 * (idx & 15);
    int du = (int)((uk[idx >> 4] >> sh) & 3u) - 1;
    int dv = (int)((vk[idx >> 4] >> sh) & 3u) - 1;
    const int neg = (du < 0) | ((du == 0) & (dv < 0));
    du = neg ? -du : du;
    dv = neg ? -dv : dv;
    const int code = du * 5 + dv;   // (0, 0) -> 0, (0, 1) -> 1 ... (2, 2) -> 12: slot + 1
    return neg ? -code : code;
}
// the joint table from A' and R' (affine): nine additions through ONE addition body.  Start points are A', R', the
// previous sum or -A'; operands are entries already written (A', R', 2R'), possibly negated.
KB_FN void ge_build_joint_table(ge_cached* tbl, const kb_half_rec& rec)
{
    ge_p3 m;
    m.X = rec.ax; m.Y = rec.ay; m.T = rec.at; fe_set(m.Z, 1);
    ge_to_cached(tbl[0], m);
    m.X = rec.rx; m.Y = rec.ry; m.T = rec.rt;
    ge_to_cached(tbl[4], m);
    ge_cached_identity(tbl[7]);
    //  step        0     1     2     3      4     5      6      7       8
    //  sum        2A'   2R'   R'+A' R'+2A' R'-A' R'-2A' 2R'+A' 2R'+2A' 2R'-A'
    //  start      A'    R'    R'    prev   R'    prev   A'     prev    -A'
    //  operand    A'    R'    A'    A'     -A'   -A'    2R'    A'      2R'
    KB_NOUNROLL
    for (int st = 0; st < 9; st++) {
        const uint32_t from = (uint32_t)(0x320212110ull >> (4 * st)) & 15u;   // 0 A', 1 R', 2 previous sum, 3 -A'
        const uint32_t opnd = (uint32_t)(0x909000040ull >> (4 * st)) & 15u;   // slot of the operand
        const uint32_t neg = (0x030u >> st) & 1u;
        const uint32_t dst = (uint32_t)(0x8BA236591ull >> (4 * st)) & 15u;
        ge_p3 b = m;
        if (from != 2) {
            const uint32_t isr = (uint32_t)(from == 1);
            b.X = rec.ax; b.Y = rec.ay; b.T = rec.at;
            fe_cmov(b.X, rec.rx, isr);
            fe_cmov(b.Y, rec.ry, isr);
            fe_cmov(b.T, rec.rt, isr);
            fe_set(b.Z, 1);
            if (from == 3) { fe_neg(b.X, b.X); fe_neg(b.T, b.T); }
        }
        ge_cached c = tbl[opnd];
        ge_cached_cneg(c, neg);
        ge_add<true>(m, b, c);
        ge_to_cached(tbl[dst], m);
    }
}
KB_FN void sig_half_setup_joint(kb_comb_digit* dw, uint32_t* uk, uint32_t* vk, ge_cached* tbl, const kb_half_rec& rec)
{
    sc_recode_comb(dw, rec.w);
    sc_joint4_bias(uk, rec.u);
    sc_joint4_bias(vk, rec.v);
    ge_build_joint_table(tbl, rec);
}
// operand of an addition, one step ahead: a joint-table entry by its code, or comb position p
KB_FN void kb_operand_fetch_code(kb_operand& o, int d, const ge_cached* tbl)
{
    o.neg = (uint32_t)d >> 31;
    const int babs = (d ^ -(int)o.neg) + (int)o.neg;
    o.nz = (uint32_t)(babs != 0);
    o.c = tbl[babs != 0 ? babs - 1 : 0];   // code = slot + 1; always a valid entry: the load is unconditional
}
KB_FN void kb_operand_fetch_comb(kb_operand& o, int p, const kb_comb_digit* dw, const ge_precomp* comb)
{
    const int d = dw[p];
    o.neg = (uint32_t)d >> 31;
    const int babs = (d ^ -(int)o.neg) + (int)o.neg;
    o.nz = (uint32_t)(babs != 0);
    kb_ld_precomp(o.c, comb + (size_t)p * KB_COMB_HALF + (babs != 0 ? babs - 1 : 0));
}
// number of radix-4 digit pairs the joint loop needs for (u, v): digits lie in [-1, 2], so n pairs represent every
// magnitude up to 2 (4^n - 1) / 3 and 2 n >= bits + 1 is enough
KB_FN int sc_joint4_pairs(const uint32_t* u, const uint32_t* v)
{
    const int bu = kb_bitlen8(u), bv = kb_bitlen8(v);
    return (bu > bv ? bu : bv) / 2 + 1;
}
// W = |v|*A' + u*R' + w*B: `npair` steps of (two doublings, one joint addition) — the first one IS its operand —
// then the comb.  The trip count is uniform over the block (the loop holds the lockstep barrier, every second pair).
// Operands are fetched one step ahead as in ge_triple_scalarmult_prefetch.
#ifndef KB_JOINT_SYNC
#define KB_JOINT_SYNC 1   // lockstep barrier when (pair index & KB_JOINT_SYNC) == KB_JOINT_SYNC: every second pair
#endif
KB_FN void ge_triple_scalarmult_joint(ge_p3& h, int npair, const kb_comb_digit* dw, const uint32_t* uk, const uint32_t* vk, const ge_cached* tbl, const ge_precomp* comb)
{
    if (npair < 2) npair = 2;   // a leading zero pair costs nothing wrong; it lets the first step below drop T
    kb_operand nx;
    kb_operand_fetch_code(nx, sc_joint4_code(uk, vk, npair - 1), tbl);
    {
        // the first addition would add to the identity: take the operand itself, (2X : 2Y : 2Z) from (Y+X, Y-X, Z);
        // doublings follow, so T is not needed
        ge_cached c;
        kb_operand_use(c, nx, false);
        fe_sub(h.X, c.YpX, c.YmX);
        fe_add(h.Y, c.YpX, c.YmX);
        fe_dbl(h.Z, c.Z);
        fe_set(h.T, 0);
    }
    KB_NOUNROLL
    for (int i = npair - 2; i >= -KB_COMB_POS; i--) {
        if (i < 0 || (i & KB_JOINT_SYNC) == KB_JOINT_SYNC) KB_LOCKSTEP();
        const int lead = i >= 0 ? 2 : 0;
        KB_NOUNROLL
        for (int step = 0; step <= lead; step++) {
            fe e, f, g, hh;
            bool with_t;
            if (step < lead) {
                ge_dbl_front(e, f, g, hh, h);
                with_t = step == lead - 1;   // the addition follows
                if (with_t) kb_operand_fetch_code(nx, sc_joint4_code(uk, vk, i), tbl);
            } else {
                ge_cached c;
                kb_operand_use(c, nx, i < 0);
                ge_add_front_z(e, f, g, hh, h, c, i < 0);   // comb entries are affine
                // T is dead when a doubling (or the end) follows: it is needed in front of the comb additions only
                with_t = i <= 0 && i != -KB_COMB_POS;
                if (with_t) kb_operand_fetch_comb(nx, -i, dw, comb);   // position -1 - (i - 1)
            }
            ge_tail(h, e, f, g, hh, with_t);
        }
    }
}
// h = a * B for a PUBLIC scalar through the comb: KB_COMB_POS (15) mixed additions instead of 64 (ge_scalarmult_base), no doublings.
// Any 32-byte scalar gives the reference's result: sc_effective is the integer the reference's digit loop
// multiplies by (SURVEY §A3), and B has order L, so that integer may be reduced mod L first.
KB_FN void ge_scalarmult_base_comb(ge_p3& h, const uint32_t* s, const ge_precomp* comb)
{
    uint32_t x[16], r[8], neg;
    sc_effective(x, neg, s);
    KB_UNROLL
    for (int i = 8; i < 16; i++) x[i] = 0;
    sc_reduce512(r, x);
    kb_comb_digit dw[KB_COMB_POS];
    sc_recode_comb(dw, r);
    ge_identity(h);
    KB_NOUNROLL
    for (int p = 0; p < KB_COMB_POS; p++) {
        const int d = dw[p];
        const uint32_t dn = (uint32_t)d >> 31;
        const int babs = (d ^ -(int)dn) + (int)dn;
        ge_cached c;
        ge_cached_identity(c);
        if (babs != 0) kb_ld_precomp(c, comb + (size_t)p * KB_COMB_HALF + (babs - 1));
        ge_precomp q;
        q.ypx = c.YpX;
        q.ymx = c.YmX;
        q.xy2d = c.T2d;
        ge_precomp_cneg(q, dn ^ neg);   // a negative multiplier negates every term
        ge_madd<true>(h, h, q);
    }
}
// comb[p][j] = (j+1) * 2^(KB_COMB_BITS p) * B in affine (y+x, y-x, 2dxy) form; entries whose multiplier does not fit 255 bits are
// never addressed by a scalar below 2^253 and hold the identity.  `base` = the 64 x 8 fixed-base table (kb_base_window).
KB_FN void kb_comb_entry(ge_precomp& out, int p, int j, const ge_precomp* base)
{
    uint32_t s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const int bit = KB_COMB_BITS * p, wi = bit >> 5, sh = bit & 31;
    const uint64_t m = (uint64_t)(j + 1) << sh;
    ge_precomp_identity(out);
    if (bit + KB_COMB_BITS + 1 > 255 && ((uint64_t)(j + 1) >> (255 - bit)) != 0) return;
    s[wi] = (uint32_t)m;
    if (wi + 1 < 8) s[wi + 1] = (uint32_t)(m >> 32);
    int8_t e[64];
    sc_recode16(e, s);
    ge_p3 h;
    ge_scalarmult_base<false>(h, e, base);
    const fe d2 = KB_FE_D2;
    fe zinv, x, y, xy;
    fe_invert(zinv, h.Z);
    fe_mul(x, h.X, zinv);
    fe_mul(y, h.Y, zinv);
    fe_add(out.ypx, y, x);
    fe_sub(out.ymx, y, x);
    fe_mul(xy, x, y);
    fe_mul(out.xy2d, xy, d2);
}
// the identity is (0 : Z : Z)
template <bool SCHNORR>
KB_FN uint32_t sig_half_finish(uint32_t f, const ge_p3& W)
{
    if (f & KB_F_FAST) {
        fe d;
        fe_sub(d, W.Y, W.Z);
        if (fe_is_zero(W.X) & fe_is_zero(d)) return KB_SIG_OK;
    }
    return sig_classify<SCHNORR>(f, (f & KB_F_ROK) ? 1u : 0u);
}
// one signature start to finish — the composition k_verify_half implements
template <bool SCHNORR>
KB_FN uint32_t sig_verify_half(const uint32_t* pk_w, const uint32_t* sig_w, const uint8_t* msg, uint64_t mlen, const ge_precomp* comb, ge_cached* tbl, int min_windows = KB_HALF_MIN_WINDOWS)
{
    kb_half_rec rec;
    sig_half_prep<SCHNORR>(rec, pk_w, sig_w, msg, mlen);
    kb_comb_digit dw[KB_COMB_POS];
    const int nwin = rec.nwin < min_windows ? min_windows : rec.nwin;
    ge_p3 W;
#if KB_HALF_JOINT
    uint32_t uk[8], vk[8];
    sig_half_setup_joint(dw, uk, vk, tbl, rec);
    const int np = sc_joint4_pairs(rec.u, rec.v);
    ge_triple_scalarmult_joint(W, np < 2 * min_windows ? 2 * min_windows : np, dw, uk, vk, tbl, comb);
#else
    int8_t eu[64], ev[64];
    sig_half_setup(dw, eu, ev, tbl, rec);
    ge_triple_scalarmult_prefetch(W, nwin, dw, eu, ev, tbl, comb);
#endif
    return sig_half_finish<SCHNORR>(rec.f, W);
}

// ---------------------------------------------------------------------------------------
// base-point table construction (replaces the transcribed BASE table, constants.rs:89)
// ---------------------------------------------------------------------------------------
// win[j] = (j+1) * pos in affine (y+x, y-x, 2dxy) form, j = 0..count-1
KB_FN void kb_base_window(ge_precomp* win, const ge_p3& pos, int count = 8)
{
    const fe d2 = KB_FE_D2;
    ge_cached pc;
    ge_to_cached(pc, pos);
    ge_p3 m = pos;
    KB_NOUNROLL
    for (int j = 0; j < count; j++) {
        fe zinv, x, y, xy;
        fe_invert(zinv, m.Z);
        fe_mul(x, m.X, zinv);
        fe_mul(y, m.Y, zinv);
        fe_add(win[j].ypx, y, x);
        fe_sub(win[j].ymx, y, x);
        fe_mul(xy, x, y);
        fe_mul(win[j].xy2d, xy, d2);
        ge_add<true>(m, m, pc);
    }
}

// ---------------------------------------------------------------------------------------
// key sets: verification under registered public keys (kb_keyset_*, capi_keyset.cu)
// ---------------------------------------------------------------------------------------
// When A is known in advance, h*A needs no doublings: a comb over A, kt[p][j] = (j+1) * 2^(KB_KEY_BITS p) * A, gives it in
// KB_KEY_POS mixed additions, and s*B comes from the context's comb in KB_COMB_POS more.  Q = s*B - h*A is then exactly
// what sig_stage1 computes, and k_verify_stage2 decides compress(Q) == R bytes as for the full-length verifiers.
// The multipliers are exact integers (never reduced mod L): a key with a small-order component has order 8L, and the
// reference's h*A with h < L must stay exact for it.
#define KB_KEY_BITS 8
#define KB_KEY_POS 32
#define KB_KEY_HALF (1 << (KB_KEY_BITS - 1))            // entries per position: (j+1) for j < KB_KEY_HALF
#define KB_KEY_ENTRIES (KB_KEY_POS * KB_KEY_HALF)       // 4096 affine entries of 96 bytes: 384 KiB per key
#define KB_KEY_INV 8                                    // comb entries made affine with one shared inversion
static_assert(KB_KEY_BITS * KB_KEY_POS >= 254 && KB_KEY_BITS <= 8, "the key comb must cover 253 bits and the recoding carry; digits are int8");
static_assert(KB_KEY_HALF % KB_KEY_INV == 0, "a position is made affine in whole groups");

// The facts about a key that sig_stage1 derives from its bytes: KB_F_AC (is_canonical), KB_F_AS (small order on bytes),
// KB_F_AOK (decodes), the last one raw — sig_keyset_flags decides per signature whether the reference reaches the decode.
// A = the decoded point for a key that can be on the fast path, the identity otherwise (its comb is never read).
KB_FN uint32_t kb_key_facts(ge_p3& A, const uint32_t* pk_w)
{
    uint32_t f = 0;
    f |= pt_is_canonical(pk_w) ? KB_F_AC : 0u;
    f |= pt_is_small_order_bytes(pk_w) ? KB_F_AS : 0u;
    f |= ge_decompress(A, pk_w) ? KB_F_AOK : 0u;
    if ((f & (KB_F_AC | KB_F_AS | KB_F_AOK)) != (KB_F_AC | KB_F_AOK)) ge_identity(A);
    return f;
}
// Position p of the key comb: row[j] = (j+1) * 2^(KB_KEY_BITS p) * A in affine (y+x, y-x, 2dxy) form, j < KB_KEY_HALF, built
// by doublings and additions of A itself.  Each group of KB_KEY_INV entries is first stored projectively in place (X, Y, Z
// in the three fields) and then made affine with ONE inversion (Montgomery's trick, as kb_batch_compress does).
KB_FN void kb_key_row(ge_precomp* row, const ge_p3& A, int p)
{
    const fe d2 = KB_FE_D2;
    ge_p3 m = A;
    const int ndbl = KB_KEY_BITS * p;
    KB_NOUNROLL
    for (int k = 0; k < ndbl; k++) ge_dbl_rt(m, m, k == ndbl - 1);
    ge_cached pc;
    ge_to_cached(pc, m);
    KB_NOUNROLL
    for (int g = 0; g < KB_KEY_HALF; g += KB_KEY_INV) {
        fe pref[KB_KEY_INV];
        fe acc;
        KB_NOUNROLL
        for (int k = 0; k < KB_KEY_INV; k++) {
            if (g + k > 0) ge_add<true>(m, m, pc);   // m = (g + k + 1) * 2^(KB_KEY_BITS p) * A
            row[g + k].ypx = m.X;
            row[g + k].ymx = m.Y;
            row[g + k].xy2d = m.Z;
            if (k == 0) acc = m.Z;
            else fe_mul(acc, acc, m.Z);
            pref[k] = acc;
        }
        fe inv;
        fe_invert(inv, acc);
        KB_NOUNROLL
        for (int k = KB_KEY_INV - 1; k >= 0; k--) {
            ge_precomp& e = row[g + k];
            fe zinv, x, y, xy;
            if (k > 0) {
                fe_mul(zinv, inv, pref[k - 1]);
                fe_mul(inv, inv, e.xy2d);
            } else {
                zinv = inv;
            }
            fe_mul(x, e.ypx, zinv);
            fe_mul(y, e.ymx, zinv);
            fe_add(e.ypx, y, x);
            fe_sub(e.ymx, y, x);
            fe_mul(xy, x, y);
            fe_mul(e.xy2d, xy, d2);
        }
    }
}
// NEGATED signed radix-2^KB_KEY_BITS digits of a scalar < 2^253: nd[p] = -d[p] with d[p] in (-KB_KEY_HALF, KB_KEY_HALF], so
// that sum nd[p] 2^(KB_KEY_BITS p) = -h and every nd[p] fits an int8
KB_FN void sc_recode_key_neg(int8_t* nd, const uint32_t* s)
{
    int carry = 0;
    KB_UNROLL
    for (int p = 0; p < KB_KEY_POS; p++) {
        const int bit = KB_KEY_BITS * p, wi = bit >> 5, sh = bit & 31;
        uint32_t x = s[wi] >> sh;
        if (sh + KB_KEY_BITS > 32 && wi + 1 < 8) x |= s[wi + 1] << (32 - sh);
        const int v = (int)(x & ((1u << KB_KEY_BITS) - 1u)) + carry;
        carry = v > KB_KEY_HALF;
        nd[p] = (int8_t)((carry << KB_KEY_BITS) - v);
    }
}
// operand of one addition: d * entry, d != 0 selects row[|d| - 1]; d = 0 gives the identity and loads nothing
KB_FN void kb_operand_fetch_row(kb_operand& o, int d, const ge_precomp* row)
{
    o.neg = (uint32_t)d >> 31;
    const int babs = (d ^ -(int)o.neg) + (int)o.neg;
    o.nz = (uint32_t)(babs != 0);
    if (babs != 0) kb_ld_precomp(o.c, row + (babs - 1));
    else ge_cached_identity(o.c);
}
// Q = s*B - h*A: KB_COMB_POS additions from the context comb, then KB_KEY_POS from the key comb, all mixed (the entries are
// affine), with the operand of the next addition fetched one step ahead as in ge_triple_scalarmult_joint.
KB_FN void ge_keyset_scalarmult(ge_p3& h, const kb_comb_digit* dw, const int8_t* nd, const ge_precomp* comb, const ge_precomp* ktab)
{
    const int nstep = KB_COMB_POS + KB_KEY_POS;
    ge_identity(h);
    kb_operand nx;
    kb_operand_fetch_row(nx, dw[0], comb);
    KB_NOUNROLL
    for (int t = 0; t < nstep; t++) {
        fe e, f, g, hh;
        ge_cached c;
        kb_operand_use(c, nx, true);
        ge_add_front_z(e, f, g, hh, h, c, true);
        const int u = t + 1;
        if (u < KB_COMB_POS) kb_operand_fetch_row(nx, dw[u], comb + (size_t)u * KB_COMB_HALF);
        else if (u < nstep) kb_operand_fetch_row(nx, nd[u - KB_COMB_POS], ktab + (size_t)(u - KB_COMB_POS) * KB_KEY_HALF);
        ge_tail(h, e, f, g, hh, u < nstep);
    }
}
// byte-level flags of the signature + the facts of its key -> the KB_F_* flags sig_stage1 would produce (without KB_F_FAST)
template <bool SCHNORR>
KB_FN uint32_t sig_keyset_flags(uint32_t kf, const uint32_t* sig_w)
{
    const uint32_t* r_w = sig_w;
    const uint32_t* s_w = sig_w + 8;
    uint32_t f = kf & (KB_F_AC | KB_F_AS);
    f |= sc_is_canonical(s_w) ? KB_F_SC : 0u;
    f |= pt_is_canonical(r_w) ? KB_F_RC : 0u;
    f |= pt_is_small_order_bytes(r_w) ? KB_F_RS : 0u;
    // EdDSA never looks at A when an earlier check fails; Schnorr decodes A before is_canonical(A)
    const uint32_t pre_ok = (f & (KB_F_SC | KB_F_RC | KB_F_RS)) == (KB_F_SC | KB_F_RC);
    if (SCHNORR || (pre_ok && (f & KB_F_AC))) f |= kf & KB_F_AOK;
    return f;
}
// sig_stage1 for a registered key: kf = kb_key_facts of it, pk_w its bytes, ktab its comb.  Items off the fast path add
// identities and read no table.
template <bool SCHNORR>
KB_FN uint32_t sig_keyset_stage1(ge_p3& Q, uint32_t kf, const uint32_t* pk_w, const uint32_t* sig_w, const uint8_t* msg, uint64_t mlen, const ge_precomp* comb, const ge_precomp* ktab)
{
    const uint32_t* r_w = sig_w;
    const uint32_t* s_w = sig_w + 8;
    const uint32_t f = sig_keyset_flags<SCHNORR>(kf, sig_w);
    const uint32_t pre_ok = (f & (KB_F_SC | KB_F_RC | KB_F_RS)) == (KB_F_SC | KB_F_RC);
    const bool fast = pre_ok && (f & (KB_F_AC | KB_F_AS | KB_F_AOK)) == (KB_F_AC | KB_F_AOK);
    kb_comb_digit dw[KB_COMB_POS];
    int8_t nd[KB_KEY_POS];
    if (fast) {
        uint32_t digest[16], hk[8];
        sha512_ram(digest, r_w, pk_w, msg, mlen);
        sc_reduce512(hk, digest);
        sc_recode_comb(dw, s_w);
        sc_recode_key_neg(nd, hk);
    } else {
        for (int p = 0; p < KB_COMB_POS; p++) dw[p] = 0;
        for (int p = 0; p < KB_KEY_POS; p++) nd[p] = 0;
    }
    ge_keyset_scalarmult(Q, dw, nd, comb, ktab);
    return fast ? (f | KB_F_FAST) : f;
}

// ---------------------------------------------------------------------------------------
// key sets: scalar multiplication of a registered key, Point::mul(s, Some(A)) (kb_keyset_mul_*, capi_keyset.cu)
// ---------------------------------------------------------------------------------------
// The key comb already holds every entry of a signed radix-16 comb over A: window w needs (j+1) * 16^w * A, j = 0..7, and
// 16^w = 2^(KB_KEY_BITS p) * 16^(w & 1) with p = w / 2, so that is kt[p][j] for an even w and kt[p][16 j + 15] for an odd
// one.  s*A is then 64 mixed additions like ge_scalarmult_base: no doublings, no decompression, no per-thread table.
static_assert(KB_KEY_BITS == 8, "two radix-16 windows per key-comb position");

// ge_select_precomp over the entries row[j * stride], j = 0..7 (stride 1 or 16, public).  CT=true reads all 8 entries and
// keeps the hit with conditional moves (no digit-dependent address or branch); CT=false loads the one it needs.
template <bool CT>
KB_FN void ge_select_precomp_strided(ge_precomp& c, const ge_precomp* row, int stride, int d)
{
    const uint32_t neg = (uint32_t)d >> 31;
    const int babs = (d ^ -(int)neg) + (int)neg;
    ge_precomp_identity(c);
    ge_cached t;
    if (CT) {
        KB_NOUNROLL
        for (int j = 0; j < 8; j++) {
            const uint32_t hit = (uint32_t)(babs == j + 1);
            kb_ld_precomp(t, row + (size_t)j * stride);
            fe_cmov(c.ypx, t.YpX, hit);
            fe_cmov(c.ymx, t.YmX, hit);
            fe_cmov(c.xy2d, t.T2d, hit);
        }
    } else if (babs != 0) {
        kb_ld_precomp(t, row + (size_t)(babs - 1) * stride);
        c.ypx = t.YpX;
        c.ymx = t.YmX;
        c.xy2d = t.T2d;
    }
    ge_precomp_cneg(c, neg);
}
// h = a * A from the key comb kt of A, e = sc_recode16(a): the sum of e[w] * 16^w * A over the 64 windows, which is the
// group element ge_scalarmult gives for the same digits (the comb's multiples are exact, never reduced mod L).
template <bool CT>
KB_FN void ge_keyset_mul(ge_p3& h, const int8_t* e, const ge_precomp* ktab)
{
    ge_precomp c;
    ge_identity(h);
    KB_NOUNROLL
    for (int w = 0; w < 64; w++) {
        const int odd = w & 1;
        ge_select_precomp_strided<CT>(c, ktab + (size_t)(w >> 1) * KB_KEY_HALF + (odd ? 15 : 0), odd ? 16 : 1, e[w]);
        ge_madd<true>(h, h, c);
    }
}
// One item: h = a * A for the registered key with facts kf (kb_key_facts), bytes pk_w and comb kt.  A key without a real
// comb (small order, not canonical or not decodable: its comb holds identities) takes the path of k_mul instead, without
// the block barrier; the key is public, so the branch is too.  Returns k_mul's status: 1 (and the identity) when the key
// does not decode.
template <bool CT>
KB_FN uint32_t kb_keyset_mul_one(ge_p3& h, uint32_t kf, const uint32_t* pk_w, const int8_t* e, const ge_precomp* kt)
{
    if ((kf & (KB_F_AC | KB_F_AS | KB_F_AOK)) == (KB_F_AC | KB_F_AOK)) {
        ge_keyset_mul<CT>(h, e, kt);
        return 0;
    }
    ge_p3 p;
    if (!ge_decompress(p, pk_w)) {
        ge_identity(h);
        return 1;
    }
    ge_cached tbl[8];
    ge_build_table8(tbl, p);
    ge_scalarmult<CT, false>(h, e, tbl);
    return 0;
}
