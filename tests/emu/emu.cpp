// tests/emu/emu.cpp — HOST EMULATION of the per-thread device math.  TEST INFRASTRUCTURE ONLY.
//
// Compiles kyber-rs_b200/csrc/{fe,ge,sc,sha512,ops}.cuh with KB_HOST_EMU so that the exact
// source the GPU kernels inline (everything except the PTX carry-chain primitives, which have
// a plain-C twin next to each asm block) can be checked against the oracle on a machine with
// no GPU.  It is never linked into libkyber_b200.so and is not a CPU fallback: the product
// library has no host compute path.
#define KB_HOST_EMU 1
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <utility>
#include <vector>
#include "../../kyber-rs_b200/csrc/ops.cuh"
#include "../../kyber-rs_b200/csrc/poly.cuh"
#include "../../kyber-rs_b200/csrc/msm.cuh"
#include "../../kyber-rs_b200/csrc/dkgfd.cuh"

static void ld(uint32_t* w, const uint8_t* b, int nwords) { memcpy(w, b, 4 * nwords); }
static void st(uint8_t* b, const uint32_t* w, int nwords) { memcpy(b, w, 4 * nwords); }

static ge_precomp g_base[64 * 8];
static ge_precomp g_base128[128];
static std::vector<ge_precomp> g_comb;   // fixed-base comb of the half-size-scalar verifiers
static int g_base_ready = 0;
static void base_init()
{
    if (g_base_ready) return;
    ge_p3 pos;
    const fe bx = KB_FE_BX, by = KB_FE_BY, bt = KB_FE_BT;
    pos.X = bx; pos.Y = by; pos.T = bt; fe_set(pos.Z, 1);
    kb_base_window(g_base128, pos, 128);
    for (int w = 0; w < 64; w++) {
        kb_base_window(g_base + 8 * w, pos);
        for (int k = 0; k < 4; k++) ge_dbl<true>(pos, pos);
    }
    g_base_ready = 1;
}

extern "C" {
// op: 0 mul, 1 sq, 2 add, 3 sub, 4 invert, 5 pow22523, 6 canon(a), 7 Karatsuba, 8/9 both row orders of mul, 10/11 of sq, 12 sub (mask wrap), 13/14 both reductions of (b : a)
void emu_fe_op(int op, uint8_t* out, const uint8_t* a, const uint8_t* b)
{
    fe x, y, r;
    ld(x.v, a, 8); ld(y.v, b, 8);
    switch (op) {
    case 0: fe_mul(r, x, y); break;
    case 1: fe_sq(r, x); break;
    case 2: fe_add(r, x, y); break;
    case 3: fe_sub(r, x, y); break;
    case 4: fe_invert(r, x); break;
    case 5: fe_pow22523(r, x); break;
    case 7: fe_mul_karatsuba(r, x, y); break;
    case 8: fe_mul_rows(r, x, y); break;
    case 9: fe_mul_rip(r, x, y); break;
    case 10: fe_sq_rows(r, x); break;
    case 11: fe_sq_rip(r, x); break;
    case 13:
    case 14: {   // both reductions of the 512-bit value (b : a): with the multiplications by 38 / by shifts (KB_FE_FOLD_SHIFT)
        uint32_t t[16];
        for (int i = 0; i < 8; i++) { t[i] = x.v[i]; t[8 + i] = y.v[i]; }
        if (op == 13) fe_reduce512_mul(r, t); else fe_reduce512_shift(r, t);
        break;
    }
    case 12: {   // fe_sub with the borrow-mask wrap (KB_FE_SUBMASK)
        uint32_t m = kb_sub8m(r.v, x.v, y.v);
        m = kb_sub_smallm(r.v, m & 38u);
        r.v[0] -= m & 38u;
        break;
    }
    default: r = x; break;
    }
    uint32_t w[8];
    fe_to_words(w, r);
    st(out, w, 8);
}
int emu_point_recode(uint8_t* out, const uint8_t* in)
{
    uint32_t w[8], o[8];
    ge_p3 p;
    ld(w, in, 8);
    uint32_t ok = ge_decompress(p, w);
    ge_compress(o, p);
    st(out, o, 8);
    return (int)ok;
}
void emu_limbs_tobytes(uint8_t* out, const int32_t* limbs)
{
    ge_p3 p;
    uint32_t o[8];
    fe_from_ref10(p.X, limbs);
    fe_from_ref10(p.Y, limbs + 10);
    fe_from_ref10(p.Z, limbs + 20);
    ge_compress(o, p);
    st(out, o, 8);
}
int emu_point_checks(const uint8_t* in)  // bit0 canonical, bit1 small-order(bytes)
{
    uint32_t w[8];
    ld(w, in, 8);
    return (int)(pt_is_canonical(w) | (pt_is_small_order_bytes(w) << 1));
}
int emu_mul(uint8_t* out, const uint8_t* scalar, const uint8_t* point, int ct)
{
    uint32_t s[8], w[8], o[8];
    ge_p3 p, h;
    ge_cached tbl[8];
    int8_t e[64];
    ld(s, scalar, 8); ld(w, point, 8);
    uint32_t ok = ge_decompress(p, w);
    sc_recode16(e, s);
    ge_build_table8(tbl, p);
    if (ct) ge_scalarmult<true>(h, e, tbl); else ge_scalarmult<false>(h, e, tbl);
    ge_compress(o, h);
    st(out, o, 8);
    return (int)ok;
}
// the joint radix-4 machinery of the half-size-scalar verifier (ops.cuh): codes[i] = sc_joint4_code of digit pair i of
// (u, v), i < 128; table[12 x 32] = encodings of the joint table built from the points a and r (slot 7 is unused)
void emu_joint4(int8_t* codes, uint8_t* table, const uint8_t* u, const uint8_t* v, const uint8_t* a, const uint8_t* r)
{
    uint32_t uw[8], vw[8], uk[8], vk[8], aw[8], rw[8];
    ld(uw, u, 8); ld(vw, v, 8); ld(aw, a, 8); ld(rw, r, 8);
    sc_joint4_bias(uk, uw);
    sc_joint4_bias(vk, vw);
    for (int i = 0; i < 128; i++) codes[i] = (int8_t)sc_joint4_code(uk, vk, i);
    ge_p3 pa, pr;
    ge_decompress(pa, aw);
    ge_decompress(pr, rw);
    kb_half_rec rec;
    rec.ax = pa.X; rec.ay = pa.Y; rec.at = pa.T;
    rec.rx = pr.X; rec.ry = pr.Y; rec.rt = pr.T;
    ge_cached tbl[KB_JOINT_SLOTS];
    ge_build_joint_table(tbl, rec);
    for (int k = 0; k < KB_JOINT_SLOTS; k++) {
        // cached (Y+X, Y-X, 2dT, Z) -> (2X : 2Y : 2Z)
        ge_p3 q;
        uint32_t o[8];
        fe_sub(q.X, tbl[k].YpX, tbl[k].YmX);
        fe_add(q.Y, tbl[k].YpX, tbl[k].YmX);
        fe_dbl(q.Z, tbl[k].Z);
        fe_set(q.T, 0);
        ge_compress(o, q);
        st(table + 32 * k, o, 8);
    }
}
void emu_mul_base(uint8_t* out, const uint8_t* scalar, int ct)
{
    uint32_t s[8], o[8];
    ge_p3 h;
    int8_t e[64];
    base_init();
    ld(s, scalar, 8);
    sc_recode16(e, s);
    if (ct) ge_scalarmult_base<true>(h, e, g_base); else ge_scalarmult_base<false>(h, e, g_base);
    ge_compress(o, h);
    st(out, o, 8);
}
static void comb_init()
{
    base_init();
    if (!g_comb.empty()) return;
    g_comb.resize((size_t)KB_COMB_POS * KB_COMB_HALF);
    // The device computes every entry on its own (k_comb_init: one scalar multiplication and one inversion per thread);
    // a host core would need minutes for the 15 x 65536 entries, so here a position is built by repeated addition of its
    // first entry and ONE inversion (Montgomery's trick).  Same points; a sample of them is checked against kb_comb_entry.
    const fe d2 = KB_FE_D2;
    std::vector<ge_p3> run(KB_COMB_HALF);
    std::vector<fe> pre(KB_COMB_HALF);
    for (int p = 0; p < KB_COMB_POS; p++) {
        ge_precomp first;
        kb_comb_entry(first, p, 0, g_base);
        ge_identity(run[0]);
        ge_madd<true>(run[0], run[0], first);
        for (int j = 1; j < KB_COMB_HALF; j++) ge_madd<true>(run[j], run[j - 1], first);
        fe acc;
        fe_set(acc, 1);
        for (int j = 0; j < KB_COMB_HALF; j++) {
            pre[j] = acc;
            fe_mul(acc, acc, run[j].Z);
        }
        fe inv;
        fe_invert(inv, acc);
        for (int j = KB_COMB_HALF - 1; j >= 0; j--) {
            fe zinv, x, y, xy;
            fe_mul(zinv, inv, pre[j]);
            fe_mul(inv, inv, run[j].Z);
            ge_precomp& out = g_comb[(size_t)p * KB_COMB_HALF + j];
            const int bit = KB_COMB_BITS * p;
            if (bit + KB_COMB_BITS + 1 > 255 && ((uint64_t)(j + 1) >> (255 - bit)) != 0) {   // never addressed (kb_comb_entry)
                ge_precomp_identity(out);
                continue;
            }
            fe_mul(x, run[j].X, zinv);
            fe_mul(y, run[j].Y, zinv);
            fe_add(out.ypx, y, x);
            fe_sub(out.ymx, y, x);
            fe_mul(xy, x, y);
            fe_mul(out.xy2d, xy, d2);
        }
        for (int j : {1, 2, KB_COMB_HALF / 3, KB_COMB_HALF - 1}) {
            ge_precomp want;
            kb_comb_entry(want, p, j, g_base);
            const ge_precomp& got = g_comb[(size_t)p * KB_COMB_HALF + j];
            uint32_t a[8], b[8];
            fe_to_words(a, got.ypx); fe_to_words(b, want.ypx);
            bool same = memcmp(a, b, 32) == 0;
            fe_to_words(a, got.ymx); fe_to_words(b, want.ymx);
            same = same && memcmp(a, b, 32) == 0;
            fe_to_words(a, got.xy2d); fe_to_words(b, want.xy2d);
            same = same && memcmp(a, b, 32) == 0;
            if (!same) { fprintf(stderr, "emu comb: entry (%d, %d) differs from kb_comb_entry\n", p, j); abort(); }
        }
    }
}
// Point::mul(s, None) for public scalars through the shared comb
void emu_mul_base_comb(uint8_t* out, const uint8_t* scalar)
{
    uint32_t s[8], o[8];
    ge_p3 h;
    comb_init();
    ld(s, scalar, 8);
    ge_scalarmult_base_comb(h, s, g_comb.data());
    ge_compress(o, h);
    st(out, o, 8);
}
void emu_sc_reduce512(uint8_t* out, const uint8_t* in)
{
    uint32_t x[16], r[8];
    ld(x, in, 16);
    sc_reduce512(r, x);
    st(out, r, 8);
}
void emu_sc_muladd(uint8_t* out, const uint8_t* a, const uint8_t* b, const uint8_t* c)
{
    uint32_t A[8], B[8], C[8], r[8];
    ld(A, a, 8); ld(B, b, 8); ld(C, c, 8);
    sc_muladd(r, A, B, C);
    st(out, r, 8);
}
void emu_sc_invert(uint8_t* out, const uint8_t* a)
{
    uint32_t A[8], r[8];
    ld(A, a, 8);
    sc_invert(r, A);
    st(out, r, 8);
}
int emu_sc_is_canonical(const uint8_t* s)
{
    uint32_t w[8];
    ld(w, s, 8);
    return (int)sc_is_canonical(w);
}
void emu_sha512_ram(uint8_t* out, const uint8_t* r, const uint8_t* a, const uint8_t* msg, uint64_t mlen)
{
    uint32_t rw[8], aw[8], d[16];
    ld(rw, r, 8); ld(aw, a, 8);
    sha512_ram(d, rw, aw, msg, mlen);
    st(out, d, 16);
}
// EdDSA::sign composed exactly as k_sign_stage1 / k_sign_finish do it
void emu_eddsa_sign(uint8_t* sig, uint8_t* pk, const uint8_t* seed_b, const uint8_t* msg, uint64_t mlen)
{
    uint32_t seed[8], d[16], d2[16], a[8], r[8], rw[8], aw[8], h[8], s[8];
    base_init();
    ld(seed, seed_b, 8);
    sha512_prefixed<8>(d, seed, nullptr, 0);
    for (int k = 0; k < 8; k++) a[k] = d[k];
    a[0] &= 0xfffffff8u;
    a[7] = (a[7] & 0x7fffffffu) | 0x40000000u;
    sha512_prefixed<8>(d2, d + 8, msg, mlen);
    sc_reduce512(r, d2);
    int8_t e[64];
    ge_p3 p;
    sc_recode16(e, r);
    ge_scalarmult_base<true>(p, e, g_base);
    ge_compress(rw, p);
    sc_recode16(e, a);
    ge_scalarmult_base<true>(p, e, g_base);
    ge_compress(aw, p);
    sha512_ram(d, rw, aw, msg, mlen);
    sc_reduce512(h, d);
    sc_muladd(s, h, a, r);
    st(sig, rw, 8);
    st(sig + 32, s, 8);
    st(pk, aw, 8);
}
int emu_sig_verify(int schnorr, const uint8_t* pk, const uint8_t* msg, uint64_t mlen, const uint8_t* sig)
{
    uint32_t pw[8], sw[16];
    ge_cached tbl[8];
    base_init();
    ld(pw, pk, 8); ld(sw, sig, 16);
    return schnorr ? (int)sig_verify<true>(pw, sw, msg, mlen, g_base128, tbl) : (int)sig_verify<false>(pw, sw, msg, mlen, g_base128, tbl);
}
// the half-size-scalar verifier (ops.cuh sig_verify_half); min_windows lets a test force longer loops
int emu_sig_verify_half(int schnorr, const uint8_t* pk, const uint8_t* msg, uint64_t mlen, const uint8_t* sig, int min_windows)
{
    uint32_t pw[8], sw[16];
    ge_cached tbl[16];
    base_init();
    ld(pw, pk, 8); ld(sw, sig, 16);
    if (min_windows < KB_HALF_MIN_WINDOWS) min_windows = KB_HALF_MIN_WINDOWS;
    comb_init();
    return schnorr ? (int)sig_verify_half<true>(pw, sw, msg, mlen, g_comb.data(), tbl, min_windows) : (int)sig_verify_half<false>(pw, sw, msg, mlen, g_comb.data(), tbl, min_windows);
}
// sc_half: out = u (32 bytes) || |v| (32 bytes); returns bits | vneg << 16
int emu_sc_half(uint8_t* out, const uint8_t* h)
{
    uint32_t hw[8];
    kb_halfsc hs;
    ld(hw, h, 8);
    sc_half(hs, hw);
    st(out, hs.u, 8);
    st(out + 32, hs.v, 8);
    return hs.bits | (int)(hs.vneg << 16);
}
// PubPoly::eval via the short-scalar Horner used by the eval kernel
int emu_pubpoly_eval(uint8_t* out, const uint8_t* commits, int t, uint32_t idx)
{
    ge_p3 v, c;
    uint32_t w[8], o[8];
    ge_identity(v);
    for (int j = t - 1; j >= 0; j--) {
        ld(w, commits + 32 * j, 8);
        if (!ge_decompress(c, w)) return 0;
        ge_cached cc;
        ge_to_cached(cc, c);
        kb_horner_step(v, (uint64_t)idx + 1, cc);
    }
    ge_compress(o, v);
    st(out, o, 8);
    return 1;
}

// The forward-difference DKG round of dkgfd.cuh for ONE dealer, with the kernels' per-cell bodies and the same
// schedule (blocks of h coefficients right-aligned in the iteration count, ping-pong arrays, n difference steps with
// the dead orders dropped, Straus combination with the host-built power table): out[i] = encoding of P(i + 1),
// i = 0..n-1.  Returns 0 if a commitment does not decode.
int emu_dkg_fd(uint8_t* out, const uint8_t* commits, int t, int n, int parts_req)
{
    size_t parts = parts_req < 1 ? 1 : (size_t)parts_req;
    if (parts > (size_t)t) parts = t;
    const size_t h = ((size_t)t + parts - 1) / parts;
    parts = ((size_t)t + h - 1) / h;
    if (parts > KB_FD_MAX_PARTS) return -1;
    std::vector<ge_p3> dec(t);
    for (int j = 0; j < t; j++) {
        uint32_t w[8];
        ld(w, commits + 32 * j, 8);
        if (!ge_decompress(dec[j], w)) return 0;
    }
    const size_t rows = parts * h;
    std::vector<ge_p3> ra(rows), rb(rows);
    const size_t hl = kb_fd_part_len(t, h, parts - 1);
    for (size_t s = 1; s < h; s++) {                // k_fd_conv, iteration s: reads src, writes dst
        std::vector<ge_p3>& src = (s & 1) ? rb : ra;
        std::vector<ge_p3>& dst = (s & 1) ? ra : rb;
        for (size_t q = 0; q < parts; q++) {
            const size_t hq = kb_fd_part_len(t, h, q);
            const size_t sq = (q + 1 < parts) ? s : (s + hl >= h ? s + hl - h : 0);
            for (size_t k = 1; k <= sq; k++) {
                ge_p3 v, lower = (k == 1) ? dec[q * h + (hq - sq)] : src[q * h + k - 1];
                const bool has_self = k < sq;
                if (has_self) v = src[q * h + k];
                kb_naf kn;
                kb_naf_from(kn, (uint64_t)k);
                kb_fd_conv_cell(v, lower, has_self, kn);
                dst[q * h + k] = v;
            }
        }
    }
    std::vector<ge_p3>& diffs = ((h - 1) & 1) ? ra : rb;
    std::vector<ge_p3> evals(parts * (size_t)n);
    for (size_t q = 0; q < parts; q++) {            // k_fd_steps, one block
        const size_t hq = kb_fd_part_len(t, h, q);
        std::vector<ge_p3> p(hq);
        p[0] = dec[q * h];
        for (size_t k = 1; k < hq; k++) p[k] = diffs[q * h + k];
        for (int i = 0; i < n; i++) {
            const size_t reach = (size_t)(n - i);
            for (size_t k = 0; k < hq; k++) {       // ascending: p[k + 1] is still the old value
                const size_t warp = k >> 5;
                if (32 * warp > reach) break;        // dead warp
                if (k + 1 < hq && 32 * ((k + 1) >> 5) <= reach) kb_fd_step_cell(p[k], p[k + 1]);
            }
            evals[q * n + i] = p[0];
        }
    }
    std::vector<uint32_t> pw(9 * (size_t)n * (parts > 1 ? parts - 1 : 1));
    kb_fd_power_table(n, h, parts, pw.data());
    const int nt = (int)parts - 1;
    for (int i = 0; i < n; i++) {                    // the combination of k_fd_check
        ge_cached tbl[8 * (KB_FD_MAX_PARTS - 1)];
        int8_t e[64 * (KB_FD_MAX_PARTS - 1)];
        ge_p3 W;
        kb_fd_combine(W, nt, pw.data() + (size_t)i * 9 * nt, tbl, e, [&](int q, ge_p3& P) { P = evals[(size_t)q * n + i]; });
        uint32_t o[8];
        ge_compress(o, W);
        st(out + 32 * i, o, 8);
    }
    return 1;
}

// the host-side table of the forward-difference round: out = n x (parts - 1) x 9 words ((i+1)^(q h) mod 8L, signed form)
void emu_fd_power_table(uint32_t* out, int n, int h, int parts) { kb_fd_power_table((size_t)n, (size_t)h, (size_t)parts, out); }
// a point given as the reference's 40 limbs: 1 and its encoding if it is a consistent curve point, else 0
int emu_point_from_limbs_checked(uint8_t* out, const int32_t* limbs)
{
    ge_p3 p;
    if (!kb_point_from_limbs_checked(p, limbs)) return 0;
    uint32_t o[8];
    ge_compress(o, p);
    st(out, o, 8);
    return 1;
}

// Pippenger stage bodies of msm.cuh, run "thread by thread" on the host; the final
// warp-shuffle tree (GPU only) is replaced by a plain sum of the same group partials.
// c, k, groups: 0 = what the driver (capi_msm.cu) picks for n points; groups is the context's KB_MSM_GROUPS setting.
int emu_msm_plan(uint8_t* out, size_t n, const uint8_t* scalars, const uint8_t* points, int c_override, int k_override, int groups_setting)
{
    kb_msm_plan pl;
    pl.n = (uint32_t)n;
    pl.c = c_override ? (uint32_t)c_override : kb_msm_window_bits_host(n);
    pl.windows = (257 + pl.c - 1) / pl.c;
    pl.half = 1u << (pl.c - 1);
    pl.nb = pl.windows * pl.half;
    pl.k = k_override ? (uint32_t)k_override : kb_msm_chunk_entries(n, pl.half);
    const uint32_t groups = kb_msm_groups_host(pl.half, (uint32_t)groups_setting);
    const size_t nthreads = (n * pl.windows + pl.k - 1) / pl.k;
    std::vector<uint32_t> pts(24 * n + 24), mags(8 * n + 8), counts(pl.nb, 0), offsets(pl.nb + 1), cursor(pl.nb, 0), sorted(n * pl.windows + 1);
    std::vector<uint32_t> bucket_sum(32 * (size_t)pl.nb), heads(32 * nthreads + 32), tails(32 * nthreads + 32), partial(32 * (size_t)pl.windows * groups);
    std::vector<uint8_t> negs(n + 1), flags(nthreads + 1);
    uint32_t bad = 0;
    for (size_t i = 0; i < n; i++) {
        uint32_t pw[8], sw[8];
        ld(pw, points + 32 * i, 8); ld(sw, scalars + 32 * i, 8);
        kb_msm_prepare_body(i, pw, sw, pts.data(), mags.data(), negs.data(), &bad);
    }
    for (size_t i = 0; i < n; i++) kb_msm_hist_body(pl, i, mags.data(), counts.data());
    uint32_t run = 0;
    for (uint32_t b = 0; b < pl.nb; b++) { offsets[b] = run; run += counts[b]; }
    offsets[pl.nb] = run;
    for (size_t i = 0; i < n; i++) kb_msm_scatter_body(pl, i, mags.data(), negs.data(), offsets.data(), cursor.data(), sorted.data());
    std::vector<uint32_t> tailb(nthreads);
    for (size_t t = 0; t < nthreads; t++) kb_msm_accum_body(pl, t, offsets.data(), sorted.data(), pts.data(), bucket_sum.data(), heads.data(), tails.data(), flags.data(), tailb.data());
    for (size_t t = 0; t < nthreads; t++) kb_msm_merge_body(pl, t, nthreads, offsets.data(), 0xffffffffu, nullptr, nullptr, bucket_sum.data(), heads.data(), tails.data(), flags.data(), tailb.data());
    std::vector<uint32_t> part_tot(32 * (size_t)pl.windows * groups);
    for (size_t t = 0; t < (size_t)pl.windows * groups; t++) kb_msm_reduce_body(pl, t, groups, offsets.data(), bucket_sum.data(), partial.data(), part_tot.data());
    // window sums as k_msm_window_sums forms them: 256 "threads" per window, chunked groups
    const uint32_t gs = (pl.half + groups - 1) / groups;
    ge_p3 tot;
    ge_identity(tot);
    for (uint32_t w = pl.windows; w-- > 0;) {
        for (uint32_t k = 0; k < pl.c; k++) ge_dbl<true>(tot, tot);
        ge_p3 a, b;
        ge_identity(a);
        ge_identity(b);
        const uint32_t per = (groups + 255) / 256;
        for (uint32_t th = 0; th < 256; th++) {
            uint32_t c0 = th * per, c1 = c0 + per;
            if (c0 > groups) c0 = groups;
            if (c1 > groups) c1 = groups;
            ge_p3 t1, t2;
            kb_msm_window_chunk(t1, t2, c0, c1, partial.data() + 32 * (size_t)w * groups, part_tot.data() + 32 * (size_t)w * groups);
            ge_cached pc;
            ge_to_cached(pc, t1);
            ge_add<true>(a, a, pc);
            ge_to_cached(pc, t2);
            ge_add<true>(b, b, pc);
        }
        ge_cached ac;
        ge_to_cached(ac, a);
        kb_horner_step(b, (uint64_t)gs, ac);
        ge_cached bc;
        ge_to_cached(bc, b);
        ge_add<true>(tot, tot, bc);
    }
    uint32_t o[8];
    ge_compress(o, tot);
    st(out, o, 8);
    return (int)bad;
}
int emu_msm(uint8_t* out, size_t n, const uint8_t* scalars, const uint8_t* points, int c_override, int k_override)
{
    return emu_msm_plan(out, n, scalars, points, c_override, k_override, 0);
}
}
