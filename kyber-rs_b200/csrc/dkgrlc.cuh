// dkgrlc.cuh — the share checks of a DKG round as ONE random linear combination per dealer (KB_ROUND_CHECK_BATCHED,
// DESIGN §3.10).
//
// Dealer d passes verifier i's check iff eval_d(x_i) == s_(d,i) B, x_i = i + 1 (vss/pedersen/vss.rs:899-912).  Write every
// commitment as C_j = P_j + tau_j (P_j of order L, tau_j in E[8]).  The reference's PubPoly::eval multiplies by the exact
// integer x, so eval(x) = sum_j x^j P_j + sum_j (x^j mod 8) tau_j, and the two parts are checked separately:
//   prime part   with weights z_i < 2^128 drawn per call:  w_j = sum_i z_i x_i^j mod L (shared by every dealer),
//                S_d = sum_i z_i s_(d,i) mod L, and  [8](sum_j w_j C_(d,j) - S_d B) = O.  [8] removes every torsion
//                component; a dealer with a wrong share passes with probability at most 2^-128.
//   torsion part exactly: x^j mod 8 is 1 (j even) and x mod 8 (j odd) for odd x; 1, x, x^2 mod 8, then 0 for even x.  So
//                A_even = sum_(j even) C_j, A_odd = sum_(j odd) C_j, C_0, C_1 and C_2 decide it for every x.  [L] kills
//                the prime part and multiplies a torsion point by 5 (L = 5 mod 8), which is invertible mod 8: a
//                combination of the [L] images vanishes iff the same combination of the torsion parts does.  The result
//                is ok_d, one bit per residue of x mod 8.
// A dealer that passes gets verdict ok_d[(i + 1) mod 8] for every i; one that fails, or has a share with byte 31 > 127
// (the reference's base multiplication need not give s B for it, ge.cuh sc_recode16), is checked share by share.
//
// The multi-scalar multiplication sum_j w_j C_(d,j) is Pippenger with signed radix-256 digits.  Its scalars are the same
// for every dealer, so the digits and, per window, the order of the j by bucket are computed once; a thread is one
// (window, chunk of that order, dealer), the 32 lanes of a warp are 32 dealers that perform the same additions.  A
// chunk walks its entries by bucket from the top down keeping `run` (the sum of its points in the buckets at or above
// the current one) and adding `run` into `tot` when it leaves a bucket, so no bucket array is stored:
//     tot + (b_bot - 1) run  =  sum over its points of bucket(p) * (+-C_p).
#pragma once
#include "ops.cuh"
#include "poly.cuh"
#include "dkgfd.cuh"

#define KB_RC_WINDOWS 32    // signed radix-256 digits of a weight < L < 2^253: window 31 takes at most 5 bits + a carry
#define KB_RC_BUCKETS 128   // digits in [-127, 128]
#define KB_RC_POW_J 32      // weights accumulated per thread of k_rc_weights

struct kb_rc_seed {
    uint32_t w[8];
};

// ---- per-thread bodies (KB_FN: also compiled by the host emulation of tests/emu) ------------------------------
// z_i = the first 16 bytes of SHA-512(seed || i || 0^24): 32 seed bytes (256 bits drawn from the OS per call), i as 8
// little-endian bytes, 24 zero bytes; z8[4..8) = 0
KB_FN void kb_rc_z(uint32_t* z8, const kb_rc_seed& seed, uint64_t i)
{
    uint32_t head[16], dg[16];
    KB_UNROLL
    for (int k = 0; k < 16; k++) head[k] = k < 8 ? seed.w[k] : 0u;
    head[8] = (uint32_t)i;
    head[9] = (uint32_t)(i >> 32);
    sha512_prefixed<16>(dg, head, nullptr, 0);
    KB_UNROLL
    for (int k = 0; k < 8; k++) z8[k] = k < 4 ? dg[k] : 0u;
}
// r = z x^e mod L (square and multiply over the public exponent e)
KB_FN void kb_rc_pow_times(uint32_t* r, const uint32_t* z8, uint64_t x, uint64_t e)
{
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t xw[8] = {(uint32_t)x, (uint32_t)(x >> 32), 0, 0, 0, 0, 0, 0}, p[8] = {1, 0, 0, 0, 0, 0, 0, 0};
    KB_NOUNROLL
    for (int b = 63; b >= 0; b--) {
        if ((e >> b) == 0) continue;
        sc_muladd(p, p, p, zero);
        if ((e >> b) & 1u) sc_muladd(p, p, xw, zero);
    }
    sc_muladd(r, p, z8, zero);
}
// w = sum_k acc[k] 2^(32 k) mod L; acc[k] < 2^64 - 2^32 (sums of at most 2^32 words)
KB_FN void kb_rc_weight(uint32_t* w, const uint64_t* acc)
{
    uint32_t x[16];
    uint64_t carry = 0;
    KB_UNROLL
    for (int k = 0; k < 8; k++) {
        const uint64_t v = acc[k] + carry;
        x[k] = (uint32_t)v;
        carry = v >> 32;
    }
    x[8] = (uint32_t)carry;
    KB_UNROLL
    for (int k = 9; k < 16; k++) x[k] = 0;
    sc_reduce512(w, x);
}
// signed radix-256 digits of w < 2^253: e[k] in [-127, 128], w = sum_k e[k] 256^k
KB_FN void kb_rc_recode256(int16_t* e, const uint32_t* w)
{
    int carry = 0;
    KB_UNROLL
    for (int k = 0; k < KB_RC_WINDOWS; k++) {
        const int d = (int)((w[k >> 2] >> (8 * (k & 3))) & 255u) + carry;
        carry = d > KB_RC_BUCKETS ? 1 : 0;
        e[k] = (int16_t)(d - (carry << 8));
    }
}
KB_FN uint32_t kb_rc_is_identity(const ge_p3& p)
{
    fe df;
    fe_sub(df, p.Y, p.Z);
    return fe_is_zero(p.X) & fe_is_zero(df);
}
// h = L p (public scalar)
KB_FN void kb_rc_mul_l(ge_p3& h, const ge_p3& p)
{
    const uint32_t l[8] = KB_L_WORDS;
    int8_t e[64];
    ge_cached tbl[8];
    sc_recode16(e, l);
    ge_build_table8(tbl, p);
    ge_scalarmult<false, false>(h, e, tbl);
}
// p += k q for a small k >= 0 (public)
KB_FN void kb_rc_add_times(ge_p3& p, const ge_p3& q, int k)
{
    ge_cached c;
    ge_to_cached(c, q);
    KB_NOUNROLL
    for (int r = 0; r < k; r++) ge_add<true>(p, p, c);
}
// bit r of the result: the torsion part of eval(x) vanishes for x = r (mod 8).
// tl = [L] A_even, [L] A_odd, [L] C_0, [L] C_1, [L] C_2 (the identity where the coefficient does not exist)
KB_FN uint32_t kb_rc_torsion_mask(const ge_p3* tl)
{
    uint32_t m = 0;
    KB_NOUNROLL
    for (int r = 0; r < 8; r++) {
        ge_p3 p;
        if (r & 1) {
            p = tl[0];
            kb_rc_add_times(p, tl[1], r);
        } else {
            p = tl[2];
            kb_rc_add_times(p, tl[3], r);
            kb_rc_add_times(p, tl[4], (r * r) & 7);
        }
        m |= kb_rc_is_identity(p) << r;
    }
    return m;
}
// one chunk [p0, p1) of a window's entries, sorted by bucket from the top down: tot = sum of bucket(p) * (+-C_(ent[p])).
// ent[p] = j | (digit < 0) << 31, bkt[p] = |digit|.  load(j, P) fetches C_j.
template <typename LD>
KB_FN void kb_rc_chunk(ge_p3& tot, const uint32_t* ent, const uint8_t* bkt, size_t p0, size_t p1, LD load)
{
    ge_identity(tot);
    if (p0 >= p1) return;
    ge_p3 run, P;
    ge_cached c;
    ge_identity(run);
    int b = bkt[p0];
    KB_NOUNROLL
    for (size_t p = p0; p < p1; p++) {
        const int bp = bkt[p];
        KB_NOUNROLL
        for (; b > bp; b--) {   // leaving bucket b
            ge_to_cached(c, run);
            ge_add<true>(tot, tot, c);
        }
        const uint32_t e = ent[p];
        load(e & 0x7fffffffu, P);
        ge_to_cached(c, P);
        ge_cached_cneg(c, e >> 31);
        ge_add<true>(run, run, c);
    }
    ge_to_cached(c, run);
    ge_add<true>(tot, tot, c);   // leaving the lowest bucket, b_bot = b
    if (b > 1) {
        kb_naf kn;
        kb_naf_from(kn, (uint64_t)(b - 1));
        kb_small_mul(run, kn);
        ge_to_cached(c, run);
        ge_add<true>(tot, tot, c);
    }
}
// W = sum_k 256^k sum_c part(k, c) over NW windows; load(k, c, P) fetches the result of chunk c of window k
template <int NW = KB_RC_WINDOWS, typename LD>
KB_FN void kb_rc_fold(ge_p3& W, size_t nch, LD load)
{
    ge_p3 P;
    ge_cached c;
    ge_identity(W);
    KB_NOUNROLL
    for (int k = NW - 1; k >= 0; k--) {
        if (k != NW - 1) {
            KB_NOUNROLL
            for (int b = 0; b < 8; b++) ge_dbl_rt(W, W, b == 7);
        }
        KB_NOUNROLL
        for (size_t q = 0; q < nch; q++) {
            load((size_t)k, q, P);
            ge_to_cached(c, P);
            ge_add<true>(W, W, c);
        }
    }
}
// [8](W - sb) == O
KB_FN uint32_t kb_rc_combination_ok(const ge_p3& W, const ge_p3& sb)
{
    ge_p3 nb, q;
    ge_cached c;
    ge_neg(nb, sb);
    ge_to_cached(c, nb);
    ge_add<true>(q, W, c);
    KB_UNROLL
    for (int k = 0; k < 3; k++) ge_dbl<true>(q, q);
    return kb_rc_is_identity(q);
}
// per-dealer state word of the round: bits 0..7 = ok_d (torsion mask), KB_RC_PASS, KB_RC_FALLBACK; 0 = a bad commitment
#define KB_RC_PASS 0x100u
#define KB_RC_FALLBACK 0x200u

#if !defined(KB_HOST_EMU)
#include "kernels.cuh"

// z_i and the weights: thread (chunk jc of KB_RC_POW_J weights, verifier i); the 32 lanes of a warp are 32 verifiers of the
// same chunk and sum their terms z_i x_i^j by shuffles before one 64-bit atomic per word (wacc[8 j + k] += word k).
static __global__ void __launch_bounds__(KB_THREADS) k_rc_weights(size_t n, size_t t, kb_rc_seed seed, uint32_t* z, unsigned long long* wacc)
{
    const size_t n32 = (n + 31) & ~(size_t)31;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t jc = idx / n32, i = idx % n32;
    const size_t j0 = jc * KB_RC_POW_J;
    if (j0 >= t) return;   // warp-uniform
    const bool live = i < n;
    uint32_t zz[8], y[8];
    kb_rc_z(zz, seed, i);
    if (!live) {
        KB_UNROLL
        for (int k = 0; k < 8; k++) zz[k] = 0;
    }
    if (jc == 0 && live) reinterpret_cast<uint4*>(z)[i] = make_uint4(zz[0], zz[1], zz[2], zz[3]);
    const uint64_t x = (uint64_t)i + 1;
    kb_rc_pow_times(y, zz, x, j0);
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0}, xw[8] = {(uint32_t)x, (uint32_t)(x >> 32), 0, 0, 0, 0, 0, 0};
    const size_t j1 = j0 + KB_RC_POW_J < t ? j0 + KB_RC_POW_J : t;
    KB_NOUNROLL
    for (size_t j = j0; j < j1; j++) {
        KB_UNROLL
        for (int k = 0; k < 8; k++) {
            unsigned long long a = y[k];
            KB_UNROLL
            for (int o = 16; o > 0; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o);
            if ((threadIdx.x & 31) == 0) atomicAdd(wacc + 8 * j + k, a);
        }
        sc_muladd(y, y, xw, zero);
    }
}
// w_j mod L and its digits: dig[k * t + j]
static __global__ void __launch_bounds__(KB_THREADS) k_rc_digits(size_t t, const unsigned long long* wacc, int16_t* dig)
{
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= t) return;
    uint64_t a[8];
    uint32_t w[8];
    int16_t e[KB_RC_WINDOWS];
    KB_UNROLL
    for (int k = 0; k < 8; k++) a[k] = wacc[8 * j + k];
    kb_rc_weight(w, a);
    kb_rc_recode256(e, w);
    KB_UNROLL
    for (int k = 0; k < KB_RC_WINDOWS; k++) dig[(size_t)k * t + j] = e[k];
}
// one block per window: the j with a non-zero digit, by bucket from the top down (counting sort; the order inside a
// bucket does not matter, the additions are exact)
static __global__ void __launch_bounds__(256) k_rc_sort(size_t t, const int16_t* dig, uint32_t* ent, uint8_t* bkt, uint32_t* cnt)
{
    __shared__ uint32_t cur[KB_RC_BUCKETS + 1];
    const size_t k = blockIdx.x;
    const int16_t* e = dig + k * t;
    for (int b = threadIdx.x; b <= KB_RC_BUCKETS; b += blockDim.x) cur[b] = 0;
    __syncthreads();
    for (size_t j = threadIdx.x; j < t; j += blockDim.x) {
        const int d = e[j], b = d < 0 ? -d : d;
        if (b) atomicAdd(cur + b, 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t off = 0;
        for (int b = KB_RC_BUCKETS; b >= 1; b--) {
            const uint32_t c = cur[b];
            cur[b] = off;
            off += c;
        }
        cnt[k] = off;
    }
    __syncthreads();
    for (size_t j = threadIdx.x; j < t; j += blockDim.x) {
        const int d = e[j], b = d < 0 ? -d : d;
        if (!b) continue;
        const uint32_t p = atomicAdd(cur + b, 1u);
        ent[k * t + p] = (uint32_t)j | (d < 0 ? 0x80000000u : 0u);
        bkt[k * t + p] = (uint8_t)b;
    }
}
// thread (window k, chunk c, dealer d): parts[((k nch + c) nd + d)] = the chunk's share of window k's bucket sum
static __global__ void __launch_bounds__(KB_THREADS) k_rc_msm(size_t nd, size_t t, size_t nch, const uint32_t* dec, const uint32_t* ent, const uint8_t* bkt, const uint32_t* cnt, uint32_t* parts)
{
    const size_t nd32 = (nd + 31) & ~(size_t)31;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t kc = idx / nd32, d = idx % nd32;
    if (kc >= KB_RC_WINDOWS * nch || d >= nd) return;
    const size_t k = kc / nch, c = kc % nch, m = cnt[k];
    ge_p3 r;
    kb_rc_chunk(r, ent + k * t, bkt + k * t, m * c / nch, m * (c + 1) / nch, [&](uint32_t j, ge_p3& P) { kb_load_p3_w128(P, KB_FD_AT(dec, j, d, nd)); });
    kb_store_p3_w128(parts + (kc * nd + d) * 32, r);
}
// thread (q, dealer d): tor[q nd + d] = [L] of A_even, A_odd, C_0, C_1, C_2 for q = 0 .. 4
static __global__ void __launch_bounds__(KB_THREADS) k_rc_torsion(size_t nd, size_t t, const uint32_t* dec, uint32_t* tor)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 5 * nd) return;
    const size_t q = idx / nd, d = idx % nd;
    ge_p3 P, C, h;
    ge_identity(P);
    if (q < 2) {
        ge_cached c;
        KB_NOUNROLL
        for (size_t j = q; j < t; j += 2) {
            kb_load_p3_w128(C, KB_FD_AT(dec, j, d, nd));
            ge_to_cached(c, C);
            ge_add<true>(P, P, c);
        }
    } else if (q - 2 < t) {
        kb_load_p3_w128(P, KB_FD_AT(dec, q - 2, d, nd));
    }
    kb_rc_mul_l(h, P);
    kb_store_p3_w128(tor + (q * nd + d) * 32, h);
}
// thread (part p, dealer d): spart[p nd + d] = sum of z_i s_(d,i) mod L over the part's verifiers, sflag = any share with
// byte 31 > 127.  The shares are secret: sc_muladd is branch-free and the loop count is public.
static __global__ void __launch_bounds__(KB_THREADS) k_rc_shares(size_t nd, size_t n, size_t sparts, const uint32_t* z, const uint8_t* shares, uint32_t* spart, uint32_t* sflag)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= sparts * nd) return;
    const size_t p = idx / nd, d = idx % nd;
    const size_t i0 = n * p / sparts, i1 = n * (p + 1) / sparts;
    uint32_t v[8] = {0, 0, 0, 0, 0, 0, 0, 0}, zz[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s[8], hi = 0;
    KB_NOUNROLL
    for (size_t i = i0; i < i1; i++) {
        const uint4 zi = __ldg(reinterpret_cast<const uint4*>(z) + i);
        zz[0] = zi.x;
        zz[1] = zi.y;
        zz[2] = zi.z;
        zz[3] = zi.w;
        kb_load32(s, shares, d * n + i);
        hi |= s[7] >> 31;
        sc_muladd(v, zz, s, v);
    }
    uint4* o = reinterpret_cast<uint4*>(spart + (p * nd + d) * 8);
    o[0] = make_uint4(v[0], v[1], v[2], v[3]);
    o[1] = make_uint4(v[4], v[5], v[6], v[7]);
    sflag[p * nd + d] = hi;
}
// thread = dealer: S_d, W_d by the fold over the windows, S_d B through the constant-time comb, the [8] test, the torsion
// mask; st[d] = the state word (KB_RC_PASS | ok_d, KB_RC_FALLBACK, or 0 for a dealer with a bad commitment)
static __global__ void __launch_bounds__(KB_THREADS) k_rc_dealer(size_t nd, size_t nch, size_t sparts, const uint32_t* parts, const uint32_t* tor, const uint32_t* spart, const uint32_t* sflag,
                                                                   const uint32_t* dealer_bad, const ge_precomp* table, uint32_t* st)
{
    extern __shared__ uint4 smem4[];
    ge_precomp* base = reinterpret_cast<ge_precomp*>(smem4);
    kb_stage(reinterpret_cast<uint32_t*>(base), reinterpret_cast<const uint32_t*>(table), 64 * 8 * 24);
    const size_t d = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= nd) return;   // no block barrier below
    const uint32_t one[8] = {1, 0, 0, 0, 0, 0, 0, 0};
    uint32_t S[8] = {0, 0, 0, 0, 0, 0, 0, 0}, v[8], hi = 0;
    KB_NOUNROLL
    for (size_t p = 0; p < sparts; p++) {
        const uint4* q = reinterpret_cast<const uint4*>(spart + (p * nd + d) * 8);
        const uint4 a = q[0], b = q[1];
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
        v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        sc_muladd(S, one, v, S);
        hi |= sflag[p * nd + d];
    }
    ge_p3 W, sb;
    kb_rc_fold(W, nch, [&](size_t k, size_t c, ge_p3& P) { kb_load_p3_w128(P, parts + ((k * nch + c) * nd + d) * 32); });
    int8_t es[64];
    sc_recode16(es, S);
    ge_scalarmult_base<true>(sb, es, base);
    const uint32_t pass = kb_rc_combination_ok(W, sb);
    ge_p3 tl[5];
    KB_UNROLL
    for (int q = 0; q < 5; q++) kb_load_p3_w128(tl[q], tor + ((size_t)q * nd + d) * 32);
    const uint32_t okm = kb_rc_torsion_mask(tl);
    st[d] = dealer_bad[d] ? 0u : (pass && !hi) ? (KB_RC_PASS | okm) : KB_RC_FALLBACK;
}
// verdict[d n + i] for the dealers that passed (and 0 for those with a bad commitment); the fallback overwrites the rest
static __global__ void __launch_bounds__(KB_THREADS) k_rc_verdict(size_t nd, size_t n, const uint32_t* st, uint8_t* verdict)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nd * n) return;
    const size_t d = idx / n, i = idx % n;
    const uint32_t s = st[d];
    verdict[idx] = (uint8_t)((s & KB_RC_PASS) ? (s >> ((i + 1) & 7)) & 1u : 0u);
}
// one block: list[0 .. *cnt) = the dealers in state KB_RC_FALLBACK, in order
static __global__ void __launch_bounds__(1024) k_rc_compact(size_t nd, const uint32_t* st, uint32_t* list, uint32_t* cnt)
{
    __shared__ uint32_t wsum[32];
    __shared__ uint32_t base;
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (size_t d0 = 0; d0 < nd; d0 += 1024) {
        const size_t d = d0 + threadIdx.x;
        const bool f = d < nd && (st[d] & KB_RC_FALLBACK);
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        if (lane == 0) wsum[w] = __popc(bal);
        __syncthreads();
        uint32_t off = base;
        for (unsigned q = 0; q < w; q++) off += wsum[q];
        if (f) list[off + __popc(bal & ((1u << lane) - 1u))] = (uint32_t)d;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t s = 0;
            for (unsigned q = 0; q < 32; q++) s += wsum[q];
            base += s;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *cnt = base;
}
#endif  // !KB_HOST_EMU
