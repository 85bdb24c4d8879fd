// ge.cuh — edwards25519 group elements on top of fe.cuh.
//
// Replaces src/group/edwards25519/ge.rs.  The reference juggles five coordinate systems
// (projective / extended / completed / precomputed / cached); here a point is always held
// in extended coordinates (X:Y:Z:T), x = X/Z, y = Y/Z, xy = T/Z, and the two operand
// forms for addition are kept:
//   ge_cached  (Y+X, Y-X, 2d*T, Z)   — ge.rs:99  write_cached
//   ge_precomp (y+x, y-x, 2d*x*y)    — ge.rs PreComputedGroupElement (Z = 1)
// The unified a=-1 addition law is complete on the whole curve (d is a non-square), so
// small-order / torsion-bearing inputs need no special cases; results are only observable
// through ge_compress, which is bit-identical to the reference (SURVEY §A4).
#pragma once
#include "fe.cuh"

struct ge_p3 {
    fe X, Y, Z, T;
};
struct ge_cached {
    fe YpX, YmX, T2d, Z;
};
struct ge_precomp {
    fe ypx, ymx, xy2d;
};

KB_FN void ge_identity(ge_p3& h)
{
    fe_set(h.X, 0);
    fe_set(h.Y, 1);
    fe_set(h.Z, 1);
    fe_set(h.T, 0);
}
KB_FN void ge_cached_identity(ge_cached& c)
{
    fe_set(c.YpX, 1);
    fe_set(c.YmX, 1);
    fe_set(c.T2d, 0);
    fe_set(c.Z, 1);
}
KB_FN void ge_precomp_identity(ge_precomp& c)
{
    fe_set(c.ypx, 1);
    fe_set(c.ymx, 1);
    fe_set(c.xy2d, 0);
}

// ---- the forms in which kernels hand points to each other through device memory, 8 little-endian words per coordinate:
//   extended point  X, Y, Z, T          32 words
//   cached operand  Y+X, Y-X, 2dT, Z    32 words
//   affine entry    y+x, y-x, 2dxy      24 words (the MSM's points)
// The suffix is the width of each access: _w32 moves single words (the host emulation compiles these), _w128 moves 16 bytes
// at a time.  Each site keeps the width it has; switching one changes its kernel's code and would need a measurement.
KB_FN void kb_store_p3_w32(uint32_t* o, const ge_p3& p)
{
    KB_UNROLL
    for (int k = 0; k < 8; k++) {
        o[k] = p.X.v[k];
        o[8 + k] = p.Y.v[k];
        o[16 + k] = p.Z.v[k];
        o[24 + k] = p.T.v[k];
    }
}
KB_FN void kb_load_p3_w32(ge_p3& p, const uint32_t* o)
{
    KB_UNROLL
    for (int k = 0; k < 8; k++) {
        p.X.v[k] = o[k];
        p.Y.v[k] = o[8 + k];
        p.Z.v[k] = o[16 + k];
        p.T.v[k] = o[24 + k];
    }
}
KB_FN void kb_store_precomp_w32(uint32_t* o, const ge_precomp& q)
{
    KB_UNROLL
    for (int k = 0; k < 8; k++) {
        o[k] = q.ypx.v[k];
        o[8 + k] = q.ymx.v[k];
        o[16 + k] = q.xy2d.v[k];
    }
}
KB_FN void kb_load_precomp_w32(ge_precomp& q, const uint32_t* o)
{
    KB_UNROLL
    for (int k = 0; k < 8; k++) {
        q.ypx.v[k] = o[k];
        q.ymx.v[k] = o[8 + k];
        q.xy2d.v[k] = o[16 + k];
    }
}
#if !defined(KB_HOST_EMU)
__device__ __forceinline__ void kb_load_fe(fe& f, const uint32_t* p)
{
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = q[0], b = q[1];
    f.v[0] = a.x; f.v[1] = a.y; f.v[2] = a.z; f.v[3] = a.w;
    f.v[4] = b.x; f.v[5] = b.y; f.v[6] = b.z; f.v[7] = b.w;
}
__device__ __forceinline__ void kb_store_fe(uint32_t* p, const fe& f)
{
    uint4* q = reinterpret_cast<uint4*>(p);
    q[0] = make_uint4(f.v[0], f.v[1], f.v[2], f.v[3]);
    q[1] = make_uint4(f.v[4], f.v[5], f.v[6], f.v[7]);
}
__device__ __forceinline__ void kb_store_p3_w128(uint32_t* o, const ge_p3& p)
{
    kb_store_fe(o, p.X);
    kb_store_fe(o + 8, p.Y);
    kb_store_fe(o + 16, p.Z);
    kb_store_fe(o + 24, p.T);
}
__device__ __forceinline__ void kb_load_p3_w128(ge_p3& p, const uint32_t* o)
{
    kb_load_fe(p.X, o);
    kb_load_fe(p.Y, o + 8);
    kb_load_fe(p.Z, o + 16);
    kb_load_fe(p.T, o + 24);
}
// the parts of an extended point that a reader needs, in the order it reads them
__device__ __forceinline__ void kb_load_p3_xy_w128(fe& x, fe& y, const uint32_t* o)
{
    kb_load_fe(x, o);
    kb_load_fe(y, o + 8);
}
__device__ __forceinline__ void kb_load_p3_z_w128(fe& z, const uint32_t* o) { kb_load_fe(z, o + 16); }
__device__ __forceinline__ void kb_store_cached_w128(uint32_t* o, const ge_cached& c)
{
    kb_store_fe(o, c.YpX);
    kb_store_fe(o + 8, c.YmX);
    kb_store_fe(o + 16, c.T2d);
    kb_store_fe(o + 24, c.Z);
}
__device__ __forceinline__ void kb_load_cached_w128(ge_cached& c, const uint32_t* o)
{
    kb_load_fe(c.YpX, o);
    kb_load_fe(c.YmX, o + 8);
    kb_load_fe(c.T2d, o + 16);
    kb_load_fe(c.Z, o + 24);
}
__device__ __forceinline__ void kb_store_precomp_w128(uint32_t* o, const ge_precomp& q)
{
    kb_store_fe(o, q.ypx);
    kb_store_fe(o + 8, q.ymx);
    kb_store_fe(o + 16, q.xy2d);
}
#endif
// ge.rs:99 write_cached
KB_FN void ge_to_cached(ge_cached& r, const ge_p3& p)
{
    const fe d2 = KB_FE_D2;
    fe_add(r.YpX, p.Y, p.X);
    fe_sub(r.YmX, p.Y, p.X);
    fe_mul(r.T2d, p.T, d2);
    r.Z = p.Z;
}
// ExtendedGroupElement::neg (ge.rs:77)
KB_FN void ge_neg(ge_p3& r, const ge_p3& p)
{
    fe_neg(r.X, p.X);
    r.Y = p.Y;
    r.Z = p.Z;
    fe_neg(r.T, p.T);
}
// -c for a cached operand: swap (Y+X, Y-X), negate 2dT
KB_FN void ge_cached_cneg(ge_cached& c, uint32_t neg)
{
    fe a = c.YpX, n;
    fe_cmov(c.YpX, c.YmX, neg);
    fe_cmov(c.YmX, a, neg);
    fe_neg(n, c.T2d);
    fe_cmov(c.T2d, n, neg);
}
KB_FN void ge_precomp_cneg(ge_precomp& c, uint32_t neg)
{
    fe a = c.ypx, n;
    fe_cmov(c.ypx, c.ymx, neg);
    fe_cmov(c.ymx, a, neg);
    fe_neg(n, c.xy2d);
    fe_cmov(c.xy2d, n, neg);
}

// r = p + q   (ge.rs:217 add + :292 to_extended; 8M).  WITH_T=false skips T3 (7M) when the
// next operation is a doubling.
KB_FN void ge_add_rt(ge_p3& r, const ge_p3& p, const ge_cached& q, bool WITH_T)
{
    fe a, b, c, d, e, f, g, h;
    fe_sub(a, p.Y, p.X);
    fe_add(b, p.Y, p.X);
    fe_mul(a, a, q.YmX);
    fe_mul(b, b, q.YpX);
    fe_mul(c, p.T, q.T2d);
    fe_mul(d, p.Z, q.Z);
    fe_dbl(d, d);
    fe_sub(e, b, a);
    fe_sub(f, d, c);
    fe_add(g, d, c);
    fe_add(h, b, a);
    fe_mul(r.X, e, f);
    fe_mul(r.Y, g, h);
    fe_mul(r.Z, f, g);
    if (WITH_T) fe_mul(r.T, e, h);
}
// r = p + q or p - q (ge.rs:217 add / :236 sub): subtraction swaps the roles of Y+X / Y-X and of
// the two sums with 2dT.  `sub` is meant to be warp-uniform (public digit of a shared scalar).
KB_FN void ge_addsub_rt(ge_p3& r, const ge_p3& p, const ge_cached& q, bool sub, bool WITH_T)
{
    fe a, b, c, d, e, f, g, h;
    fe_sub(a, p.Y, p.X);
    fe_add(b, p.Y, p.X);
    if (sub) {
        fe_mul(a, a, q.YpX);
        fe_mul(b, b, q.YmX);
    } else {
        fe_mul(a, a, q.YmX);
        fe_mul(b, b, q.YpX);
    }
    fe_mul(c, p.T, q.T2d);
    fe_mul(d, p.Z, q.Z);
    fe_dbl(d, d);
    fe_sub(e, b, a);
    if (sub) {
        fe_add(f, d, c);
        fe_sub(g, d, c);
    } else {
        fe_sub(f, d, c);
        fe_add(g, d, c);
    }
    fe_add(h, b, a);
    fe_mul(r.X, e, f);
    fe_mul(r.Y, g, h);
    fe_mul(r.Z, f, g);
    if (WITH_T) fe_mul(r.T, e, h);
}
// r = p + q with q affine-precomputed (ge.rs:274 mixed_add; 7M / 6M)
KB_FN void ge_madd_rt(ge_p3& r, const ge_p3& p, const ge_precomp& q, bool WITH_T)
{
    fe a, b, c, d, e, f, g, h;
    fe_sub(a, p.Y, p.X);
    fe_add(b, p.Y, p.X);
    fe_mul(a, a, q.ymx);
    fe_mul(b, b, q.ypx);
    fe_mul(c, p.T, q.xy2d);
    fe_dbl(d, p.Z);
    fe_sub(e, b, a);
    fe_sub(f, d, c);
    fe_add(g, d, c);
    fe_add(h, b, a);
    fe_mul(r.X, e, f);
    fe_mul(r.Y, g, h);
    fe_mul(r.Z, f, g);
    if (WITH_T) fe_mul(r.T, e, h);
}
// r = 2p   (ge.rs:35 ProjectiveGroupElement::double; 4S + 4M, or 4S + 3M without T)
KB_FN void ge_dbl_rt(ge_p3& r, const ge_p3& p, bool WITH_T)
{
    fe a, b, c, e, f, g, h;
    fe_sq(a, p.X);
    fe_sq(b, p.Y);
    fe_sq(c, p.Z);
    fe_dbl(c, c);
    fe_add(h, a, b);
    fe_add(e, p.X, p.Y);
    fe_sq(e, e);
    fe_sub(e, h, e);
    fe_sub(g, a, b);
    fe_add(f, c, g);
    fe_mul(r.X, e, f);
    fe_mul(r.Y, g, h);
    fe_mul(r.Z, f, g);
    if (WITH_T) fe_mul(r.T, e, h);
}

// The unified addition and the doubling END in the same four products (X3 = E F, Y3 = G H, Z3 = F G, T3 = E H):
// split into front ends and ONE shared tail, a loop over "steps" holds the tail's code once (the long
// scalar-multiplication kernels are bound by the instruction cache as much as by the multiplier).
KB_FN void ge_add_front(fe& e, fe& f, fe& g, fe& h, const ge_p3& p, const ge_cached& q)
{
    fe a, b, c, d;
    fe_sub(a, p.Y, p.X);
    fe_add(b, p.Y, p.X);
    fe_mul(a, a, q.YmX);
    fe_mul(b, b, q.YpX);
    fe_mul(c, p.T, q.T2d);
    fe_mul(d, p.Z, q.Z);
    fe_dbl(d, d);
    fe_sub(e, b, a);
    fe_sub(f, d, c);
    fe_add(g, d, c);
    fe_add(h, b, a);
}
// the same when the operand is known to have Z = 1 in some calls (q_z_one, uniform over the warp): 2 Z1 needs no product
KB_FN void ge_add_front_z(fe& e, fe& f, fe& g, fe& h, const ge_p3& p, const ge_cached& q, bool q_z_one)
{
    fe a, b, c, d;
    fe_sub(a, p.Y, p.X);
    fe_add(b, p.Y, p.X);
    fe_mul(a, a, q.YmX);
    fe_mul(b, b, q.YpX);
    fe_mul(c, p.T, q.T2d);
    if (q_z_one) d = p.Z;
    else fe_mul(d, p.Z, q.Z);
    fe_dbl(d, d);
    fe_sub(e, b, a);
    fe_sub(f, d, c);
    fe_add(g, d, c);
    fe_add(h, b, a);
}
KB_FN void ge_dbl_front(fe& e, fe& f, fe& g, fe& h, const ge_p3& p)
{
    fe a, b, c;
    fe_sq(a, p.X);
    fe_sq(b, p.Y);
    fe_sq(c, p.Z);
    fe_dbl(c, c);
    fe_add(h, a, b);
    fe_add(e, p.X, p.Y);
    fe_sq(e, e);
    fe_sub(e, h, e);
    fe_sub(g, a, b);
    fe_add(f, c, g);
}
KB_FN void ge_tail(ge_p3& r, const fe& e, const fe& f, const fe& g, const fe& h, bool WITH_T)
{
    fe_mul(r.X, e, f);
    fe_mul(r.Y, g, h);
    fe_mul(r.Z, f, g);
    if (WITH_T) fe_mul(r.T, e, h);
}

// compile-time flavours (the flag folds away when the call is inlined with a constant)
template <bool WITH_T = true>
KB_FN void ge_add(ge_p3& r, const ge_p3& p, const ge_cached& q) { ge_add_rt(r, p, q, WITH_T); }
template <bool WITH_T = true>
KB_FN void ge_madd(ge_p3& r, const ge_p3& p, const ge_precomp& q) { ge_madd_rt(r, p, q, WITH_T); }
template <bool WITH_T = true>
KB_FN void ge_dbl(ge_p3& r, const ge_p3& p) { ge_dbl_rt(r, p, WITH_T); }

// ExtendedGroupElement::set_bytes (ge.rs:124-179).  w = the 32-byte encoding as 8 LE words.
// Returns 1 on success.  y >= p is accepted (taken mod p); x = 0 with the sign bit set is
// accepted (SURVEY §A2).
KB_FN uint32_t ge_decompress(ge_p3& h, const uint32_t* w)
{
    const fe d = KB_FE_D;
    const fe sqrtm1 = KB_FE_SQRTM1;
    fe u, v, v3, vxx, check, x;
    fe_from_words(h.Y, w);
    fe_set(h.Z, 1);
    fe_sq(u, h.Y);
    fe_mul(v, u, d);
    fe_sub(u, u, h.Z);  // u = y^2 - 1
    fe_add(v, v, h.Z);  // v = d y^2 + 1
    fe_sq(v3, v);
    fe_mul(v3, v3, v);  // v^3
    fe_sq(x, v3);
    fe_mul(x, x, v);
    fe_mul(x, x, u);    // u v^7
    fe_pow22523(x, x);
    fe_mul(x, x, v3);
    fe_mul(x, x, u);    // u v^3 (u v^7)^((p-5)/8)
    fe_sq(vxx, x);
    fe_mul(vxx, vxx, v);
    fe_sub(check, vxx, u);
    uint32_t ok_direct = fe_is_zero(check);
    fe_add(check, vxx, u);
    uint32_t ok_twisted = fe_is_zero(check);
    fe xi;
    fe_mul(xi, x, sqrtm1);
    fe_cmov(x, xi, (ok_direct ^ 1u) & ok_twisted);
    uint32_t flip = fe_is_negative(x) ^ (w[7] >> 31);
    fe nx;
    fe_neg(nx, x);
    fe_cmov(x, nx, flip);
    h.X = x;
    fe_mul(h.T, h.X, h.Y);
    return ok_direct | ok_twisted;
}

// ExtendedGroupElement::write_bytes (ge.rs:112-122) given zinv = 1/Z
KB_FN void ge_compress_with_zinv(uint32_t* w, const ge_p3& p, const fe& zinv)
{
    fe x, y;
    fe_mul(x, p.X, zinv);
    fe_mul(y, p.Y, zinv);
    fe_to_words(w, y);
    w[7] ^= fe_is_negative(x) << 31;
}
KB_FN void ge_compress(uint32_t* w, const ge_p3& p)
{
    fe zinv;
    fe_invert(zinv, p.Z);
    ge_compress_with_zinv(w, p, zinv);
}

// ---------------------------------------------------------------------------------------
// the reference's in-memory / serde field element: 10 signed limbs, radix 2^25.5 (fe.rs:8)
// ---------------------------------------------------------------------------------------
// kyber-rs serialises a Point with serde as its raw ExtendedGroupElement (4 x 10 i32 limbs + a bool,
// 161 bytes: ge.rs:75-83, point.rs:23-27) and does not validate it on decode (SURVEY §8f-3), so any i32
// limb values must be accepted: h = sum_i l[i] * 2^ceil(25.5 i) mod p.
KB_FN void fe_from_ref10(fe& h, const int32_t* l)
{
    const int off[10] = {0, 26, 51, 77, 102, 128, 153, 179, 204, 230};
    uint32_t pos[9], neg[9];
    KB_UNROLL
    for (int k = 0; k < 9; k++) pos[k] = neg[k] = 0;
    KB_UNROLL
    for (int i = 0; i < 10; i++) {
        const int64_t v = l[i];
        const uint64_t mag = (uint64_t)(v < 0 ? -v : v);  // <= 2^31
        uint32_t* acc = v < 0 ? neg : pos;
        const int w = off[i] >> 5, sh = off[i] & 31;
        // mag << sh spans at most 3 words
        const uint64_t lo = mag << sh;
        const uint32_t hi3 = sh ? (uint32_t)(mag >> (64 - sh)) : 0u;
        uint64_t c = (uint64_t)acc[w] + (uint32_t)lo;
        acc[w] = (uint32_t)c;
        c = (c >> 32) + acc[w + 1] + (uint32_t)(lo >> 32);
        acc[w + 1] = (uint32_t)c;
        c >>= 32;
        if (w + 2 < 9) {
            c += (uint64_t)acc[w + 2] + hi3;
            acc[w + 2] = (uint32_t)c;
            c >>= 32;
            KB_UNROLL
            for (int k = w + 3; k < 9; k++) {
                c += acc[k];
                acc[k] = (uint32_t)c;
                c >>= 32;
            }
        }
    }
    // fold word 8 (2^256 = 38) of each part, then subtract
    fe a, b;
    KB_UNROLL
    for (int k = 0; k < 8; k++) {
        a.v[k] = pos[k];
        b.v[k] = neg[k];
    }
    uint32_t c1 = kb_add_small(a.v, pos[8] * 38u);
    a.v[0] += 38u * c1;
    uint32_t c2 = kb_add_small(b.v, neg[8] * 38u);
    b.v[0] += 38u * c2;
    fe_sub(h, a, b);
}

// A whole ExtendedGroupElement from its 40 limbs (X, Y, Z, T), for entry points that keep computing with it.  The
// reference never validates this form (Deal::decode, share/vss/pedersen/vss.rs:155-159) and its results on
// inconsistent limbs depend on its exact operation sequence; here an element is accepted only if it is a consistent
// representation of a curve point:  Z != 0,  T Z = X Y  and  -X^2 + Y^2 = Z^2 + d T^2.  Returns 1 if so.
KB_FN uint32_t kb_point_from_limbs_checked(ge_p3& p, const int32_t* l)
{
    fe_from_ref10(p.X, l);
    fe_from_ref10(p.Y, l + 10);
    fe_from_ref10(p.Z, l + 20);
    fe_from_ref10(p.T, l + 30);
    const fe d = KB_FE_D;
    fe a, b, xx, yy, df;
    fe_mul(a, p.T, p.Z);
    fe_mul(b, p.X, p.Y);
    fe_sub(df, a, b);
    uint32_t ok = fe_is_zero(df) & (fe_is_zero(p.Z) ^ 1u);
    fe_sq(xx, p.X);
    fe_sq(yy, p.Y);
    fe_sub(a, yy, xx);      // -X^2 + Y^2
    fe_sq(b, p.T);
    fe_mul(b, b, d);
    fe_sq(xx, p.Z);
    fe_add(b, b, xx);       // Z^2 + d T^2
    fe_sub(df, a, b);
    ok &= fe_is_zero(df);
    return ok;
}

// ---------------------------------------------------------------------------------------
// scalar recoding — the reference's signed radix-16 digits (ge.rs:443-458 / :521-535)
// ---------------------------------------------------------------------------------------
// e[0..63]: e[0..62] in [-8, 8), e[63] = top nibble + carry.  A top digit outside 0..8 (only
// possible when the documented precondition a[31] <= 127 is violated) selects nothing in
// select_pre_computed / select_cached (ge.rs:423-434, 488-500) and contributes the identity
// (SURVEY §A3); we reproduce that by zeroing it, so EVERY 32-byte scalar gives the
// reference's result.
KB_FN void sc_recode16(int8_t* e, const uint32_t* s)
{
    int carry = 0;
    KB_UNROLL
    for (int i = 0; i < 63; i++) {
        int d = (int)((s[i >> 3] >> (4 * (i & 7))) & 15u) + carry;
        carry = (d + 8) >> 4;
        e[i] = (int8_t)(d - (carry << 4));
    }
    int top = (int)(s[7] >> 28) + carry;
    e[63] = (int8_t)((top > 8) ? 0 : top);
}
