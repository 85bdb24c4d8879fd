// dkgfd.cuh — a whole DKG deal-verification round by FORWARD DIFFERENCES.
//
// The reference checks every share with its own PubPoly::eval (share/poly.rs:457-469): for dealer d and verifier
// i, a Horner run over the t commitments at x = i + 1, i.e. n * t small-scalar steps per dealer (k_poly_eval does
// exactly that).  But the n evaluation points of one dealer are CONSECUTIVE integers, and for consecutive points a
// polynomial of degree h - 1 obeys  Δ^k E(x + 1) = Δ^k E(x) + Δ^(k+1) E(x):  once the h forward differences at one
// point are known, every further evaluation costs h - 1 point ADDITIONS instead of h multiplications by x.
// Everything below is an integer-linear combination of the commitments, so it holds in any abelian group — in
// particular for commitments that carry a small-order component (SURVEY §7-H2).
//
//   0  The t commitments of a dealer are cut into `parts` blocks of h consecutive coefficients,
//          P(x) = sum_q x^(q h) E_q(x),   E_q(x) = sum_{j<h} C_(q h + j) x^j
//      (the last block may be shorter).  Shorter blocks make stage A cheaper (it is quadratic in h) and its chain of
//      dependent launches shorter; they are paid for in stage D.
//   A  Forward differences r_k = Δ^k E_q(0) by Horner's rule in the BINOMIAL basis: E = sum_k r_k C(x, k), and because
//      x C(x, k) = k C(x, k) + (k+1) C(x, k+1), multiplying by x and adding the next coefficient c is
//          r'_k = k (r_k + r_(k-1))   (k >= 1),      r'_0 = c.
//      One launch per coefficient (h - 1 launches for ALL blocks and dealers), every cell one point addition and one
//      multiplication by the small integer k < h.  No division and no factorial ever appears.
//   C  ONE launch runs all n difference steps: a thread block owns one (dealer, block), its lanes are the ORDERS k,
//      the state lives in registers for the whole run, neighbours exchange the operand by warp shuffle (and through
//      shared memory across a warp boundary); lane 0 records E_q(i + 1) after step i.
//   D  verdict(d, i) = [ E_0 + sum_q (x^(q h) mod 8L) E_q == share * B ],  x = i + 1: Straus over the parts - 1 tables with
//      shared doublings (the multipliers are public and the same for the 32 dealers of a warp), the share through the
//      constant-time fixed-base comb (shares are secret), compared projectively as k_poly_eval does
//      (vss/pedersen/vss.rs:899-912).
//
// For n = 1024, t = 683, 4 blocks this is ~0.9 x 10^9 multiplies per dealer instead of 4.75 x 10^9 (Horner per share).
#pragma once
#include "ops.cuh"
#include "poly.cuh"

#define KB_FD_MAX_PARTS 4
#define KB_FD_MAX_H 256     // orders of one block = threads of one k_fd_steps block

// ---- per-cell bodies (KB_FN: also compiled by the host emulation of tests/emu) ------------------------------
// v = k * v for a small public integer k >= 1 given by its NAF; T is valid on return
KB_FN void kb_small_mul(ge_p3& v, const kb_naf& k)
{
    if (k.len <= 1) return;
    ge_cached vc;
    ge_to_cached(vc, v);
    ge_p3 acc = v;
    KB_NOUNROLL
    for (int i = k.len - 2; i >= 0; i--) {
        const int d = k.d[i];
        ge_dbl_rt(acc, acc, d != 0 || i == 0);
        if (d != 0) ge_addsub_rt(acc, acc, vc, d < 0, i == 0);
    }
    v = acc;
}
// A: one cell of the conversion, v = k * (v + lower); with has_self == false (the order that appears in this
// iteration) v = k * lower
KB_FN void kb_fd_conv_cell(ge_p3& v, const ge_p3& lower, bool has_self, const kb_naf& k)
{
    if (has_self) {
        ge_cached c;
        ge_to_cached(c, lower);
        ge_add<true>(v, v, c);
    } else {
        v = lower;
    }
    kb_small_mul(v, k);
}
// C: p += q
KB_FN void kb_fd_step_cell(ge_p3& p, const ge_p3& q)
{
    ge_cached c;
    ge_to_cached(c, q);
    ge_add<true>(p, p, c);
}
// D: W = E_0 + sum_{q=1..nt} s_q * E_q.  load(q, P) fetches E_q; pw9 = nt x 9 words (|s_q| <= 4L as 8 words + sign);
// tbl = 8 * nt entries and e = 64 * nt digits of caller-provided scratch.
template <typename LD>
KB_FN void kb_fd_combine(ge_p3& W, int nt, const uint32_t* pw9, ge_cached* tbl, int8_t* e, LD load)
{
    ge_p3 P;
    KB_NOUNROLL
    for (int q = 0; q < nt; q++) {
        load(q + 1, P);
        if (pw9[9 * q + 8]) {
            fe_neg(P.X, P.X);
            fe_neg(P.T, P.T);
        }
        sc_recode16(e + 64 * q, pw9 + 9 * q);
        ge_build_table8(tbl + 8 * q, P);
    }
    ge_identity(W);
    if (nt > 0) {
        KB_NOUNROLL
        for (int i = 63; i >= 0; i--) {
            KB_LOCKSTEP();
            if (i != 63) {
                KB_NOUNROLL
                for (int k = 0; k < 4; k++) ge_dbl_rt(W, W, k == 3);
            }
            KB_NOUNROLL
            for (int q = 0; q < nt; q++) {
                ge_cached c;
                ge_select_cached<false>(c, tbl + 8 * q, e[64 * q + i]);
                ge_add_rt(W, W, c, q + 1 < nt || i == 0);
            }
        }
    }
    load(0, P);
    ge_cached c0;
    ge_to_cached(c0, P);
    ge_add<true>(W, W, c0);
}

// ---- host integers: the table of stage D -----------------------------------------------------------------------
// x <- x * k mod 8L for a small k (< 2^32); x = 4 x 64-bit words, < 8L
static inline void kb_mul_small_mod_8l(uint64_t* x, uint64_t k)
{
    const uint64_t N[4] = {0xc09318d2e7ae9f68ull, 0xa6f7cef517bce6b2ull, 0ull, 0x8000000000000000ull};
    uint64_t y[5];
    unsigned __int128 c = 0;
    for (int i = 0; i < 4; i++) {
        c += (unsigned __int128)x[i] * k;
        y[i] = (uint64_t)c;
        c >>= 64;
    }
    y[4] = (uint64_t)c;
    // N = 2^255 + (a 128-bit number): floor(y / 2^255) is the quotient or one more
    const uint64_t q = (y[4] << 1) | (y[3] >> 63);
    unsigned __int128 mc = 0;
    uint64_t qn[5];
    for (int i = 0; i < 4; i++) {
        mc += (unsigned __int128)N[i] * q;
        qn[i] = (uint64_t)mc;
        mc >>= 64;
    }
    qn[4] = (uint64_t)mc;
    uint64_t borrow = 0;
    for (int i = 0; i < 5; i++) {
        const unsigned __int128 dd = (unsigned __int128)y[i] - qn[i] - borrow;
        y[i] = (uint64_t)dd;
        borrow = (uint64_t)(dd >> 64) & 1u;
    }
    if (borrow) {   // one N too many: add it back
        unsigned __int128 a = 0;
        for (int i = 0; i < 5; i++) {
            a += (unsigned __int128)y[i] + (i < 4 ? N[i] : 0);
            y[i] = (uint64_t)a;
            a >>= 64;
        }
    }
    for (int i = 0; i < 4; i++) x[i] = y[i];
}
// signed representative of x mod 8L: 8 words of magnitude (<= 4L, inside the domain of the radix-16 recoding) + 1 word of sign
static inline void kb_signed_mod_8l(uint32_t* out9, const uint64_t* x)
{
    const uint64_t N[4] = {0xc09318d2e7ae9f68ull, 0xa6f7cef517bce6b2ull, 0ull, 0x8000000000000000ull};
    const uint64_t H[4] = {0x60498c6973d74fb4ull, 0x537be77a8bde7359ull, 0ull, 0x4000000000000000ull};   // N / 2 = 4L
    bool big = false;
    for (int i = 3; i >= 0; i--) {
        if (x[i] != H[i]) {
            big = x[i] > H[i];
            break;
        }
    }
    uint64_t m[4];
    if (big) {
        uint64_t borrow = 0;
        for (int i = 0; i < 4; i++) {
            const unsigned __int128 dd = (unsigned __int128)N[i] - x[i] - borrow;
            m[i] = (uint64_t)dd;
            borrow = (uint64_t)(dd >> 64) & 1u;
        }
    } else {
        for (int i = 0; i < 4; i++) m[i] = x[i];
    }
    for (int i = 0; i < 4; i++) {
        out9[2 * i] = (uint32_t)m[i];
        out9[2 * i + 1] = (uint32_t)(m[i] >> 32);
    }
    out9[8] = big ? 1u : 0u;
}
// out[(i * (parts - 1) + (q - 1)) * 9 ..] = (i + 1)^(q h) mod 8L in signed form, i < n, 1 <= q < parts.
// Host integers only (table construction, like the window counts of the MSM plan): (parts - 1) * h small
// multiplications per evaluation point.
static inline void kb_fd_power_table(size_t n, size_t h, size_t parts, uint32_t* out)
{
    if (parts < 2) return;
    for (size_t i = 0; i < n; i++) {
        uint64_t x[4] = {1, 0, 0, 0};
        for (size_t q = 1; q < parts; q++) {
            for (size_t r = 0; r < h; r++) kb_mul_small_mod_8l(x, (uint64_t)i + 1);
            kb_signed_mod_8l(out + (i * (parts - 1) + (q - 1)) * 9, x);
        }
    }
}
// length of block q when t coefficients are cut into blocks of h
#if defined(KB_HOST_EMU)
#define KB_HD static inline
#else
#define KB_HD __host__ __device__ __forceinline__
#endif
KB_HD size_t kb_fd_part_len(size_t t, size_t h, size_t q) { return (q + 1) * h <= t ? h : t - q * h; }

#if !defined(KB_HOST_EMU)
#include "kernels.cuh"

// arrays of extended points, 32 words each: row-major [row][dealer] (a warp = 32 dealers of one row)
#define KB_FD_AT(arr, row, d, nd) ((arr) + (((size_t)(row) * (nd) + (d)) * 32))
#ifndef KB_FD_CONV_THREADS
#define KB_FD_CONV_THREADS 128
#endif
#ifndef KB_FD_CONV_MINBLOCKS
#define KB_FD_CONV_MINBLOCKS 3
#endif

// dec[j][d] = commitment j of dealer d, decoded; dealer_bad[d] |= 1 if any commitment does not decode
static __global__ void __launch_bounds__(KB_THREADS) k_fd_decode(size_t nd, size_t t, const uint8_t* commits, uint32_t* dec, uint32_t* dealer_bad)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nd * t) return;
    const size_t j = idx / nd, d = idx % nd;
    uint32_t w[8];
    kb_load32(w, commits, d * t + j);
    ge_p3 p;
    if (!ge_decompress(p, w)) {
        ge_identity(p);
        atomicOr(dealer_bad + d, 1u);
    }
    kb_store_p3_w128(KB_FD_AT(dec, j, d, nd), p);
}
// The same from the reference's in-memory / serde form of a Point: X, Y, Z, T as 10 signed 25.5-bit limbs each
// (ge.rs:75-83).  That form is not validated by the reference (SURVEY §8f-3); here an element that is not a
// consistent representation of a curve point (T Z != X Y, Z = 0 or off the curve) marks its dealer bad.
static __global__ void __launch_bounds__(KB_THREADS) k_fd_decode_limbs(size_t nd, size_t t, const int32_t* limbs, uint32_t* dec, uint32_t* dealer_bad)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nd * t) return;
    const size_t j = idx / nd, d = idx % nd;
    ge_p3 p;
    if (!kb_point_from_limbs_checked(p, limbs + 40 * (d * t + j))) {
        ge_identity(p);
        atomicOr(dealer_bad + d, 1u);
    }
    kb_store_p3_w128(KB_FD_AT(dec, j, d, nd), p);
}

// Stage A, iteration s = 1 .. h-1.  Block q of a dealer has length hq; it is right-aligned in the iteration count
// (sq = s - (h - hq) is its own iteration number), so that all blocks finish together.  Its iteration sq brings in
// coefficient hq-1-sq and touches the orders k = 1 .. sq:  dst[k] = k * (src[k] + src[k-1]), where src[0] is the
// coefficient brought in by the previous iteration (read from `dec`) and src[sq] is still zero.
// Rows of src / dst: q * h + k.
static __global__ void __launch_bounds__(KB_FD_CONV_THREADS, KB_FD_CONV_MINBLOCKS) k_fd_conv(size_t nd, size_t t, size_t h, size_t parts, size_t s, const uint32_t* dec, const uint32_t* src, uint32_t* dst)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t hl = kb_fd_part_len(t, h, parts - 1);          // length of the last block
    const size_t sl = s + hl >= h ? s + hl - h : 0;            // its iteration number (0: not started)
    const size_t cells = (parts - 1) * s + sl;                  // per dealer
    if (idx >= nd * cells) return;
    // the cost of a cell grows with log2(k): the cells with the large multipliers go first, so that the launch does
    // not end on them
    const size_t c = idx / nd, d = idx % nd;
    size_t q, k, sq, hq;
    if (c < (parts - 1) * s) {
        q = c % (parts - 1);
        k = s - c / (parts - 1);
        sq = s;
        hq = h;
    } else {
        q = parts - 1;
        k = sl - (c - (parts - 1) * s);
        sq = sl;
        hq = hl;
    }
    ge_p3 v, lower;
    if (k == 1) kb_load_p3_w128(lower, KB_FD_AT(dec, q * h + (hq - sq), d, nd));
    else kb_load_p3_w128(lower, KB_FD_AT(src, q * h + k - 1, d, nd));
    const bool has_self = k < sq;
    if (has_self) kb_load_p3_w128(v, KB_FD_AT(src, q * h + k, d, nd));
    kb_naf kn;
    kb_naf_from(kn, (uint64_t)k);
    kb_fd_conv_cell(v, lower, has_self, kn);
    kb_store_p3_w128(KB_FD_AT(dst, q * h + k, d, nd), v);
}

// ---- Stage A for SMALL rounds: one cell on FOUR lanes -----------------------------------------------------------------
// With few dealers (the shard of one rank of 8, config 3) a conversion launch holds so few cells that it lasts exactly one
// cell's latency: an addition and a multiplication by k, about 12 dependent point operations of ~1 us each on a lone warp
// (a point operation is two or three levels of four independent field multiplications, and one warp cannot issue an
// IMAD.WIDE more often than every 4 cycles: 4 x 73 x 4 cycles per level).  Here the four lanes of a quad hold the same
// point and each does ONE of the four multiplications of a level; the products travel by warp shuffle.  Same formulas,
// same results (every lane ends with the full point); 2.5x shorter latency for 4x the lanes — used only while the grid
// leaves the GPU mostly idle (kb_dkg_fd_run).
// (the shuffles name only the four lanes of the quad, so the quads of a warp — which may hold cells with different
// multipliers — are free to diverge from each other)
__device__ __forceinline__ void kb_q4_bcast(fe& out, const fe& in, int src_lane)
{
    const unsigned mask = 0xFu << (src_lane & 28);
#pragma unroll
    for (int w = 0; w < 8; w++) out.v[w] = __shfl_sync(mask, in.v[w], src_lane);
}
// the closing products of the addition / doubling formulas: X3 = E F, Y3 = G H, Z3 = F G, T3 = E H
__device__ __forceinline__ void kb_q4_tail(ge_p3& p, const fe& e, const fe& f, const fe& g, const fe& h)
{
    const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
    fe l = e, r = f, prod;
    fe_cmov(l, g, (uint32_t)(role == 1));
    fe_cmov(l, f, (uint32_t)(role == 2));
    fe_cmov(r, h, (uint32_t)(role == 1 || role == 3));
    fe_cmov(r, g, (uint32_t)(role == 2));
    fe_mul(prod, l, r);
    kb_q4_bcast(p.X, prod, base + 0);
    kb_q4_bcast(p.Y, prod, base + 1);
    kb_q4_bcast(p.Z, prod, base + 2);
    kb_q4_bcast(p.T, prod, base + 3);
}
__device__ __forceinline__ void kb_q4_dbl(ge_p3& p)
{
    const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
    fe in = p.X, t, sq;
    fe_add(t, p.X, p.Y);
    fe_cmov(in, p.Y, (uint32_t)(role == 1));
    fe_cmov(in, p.Z, (uint32_t)(role == 2));
    fe_cmov(in, t, (uint32_t)(role == 3));
    fe_sq(sq, in);
    fe a, b, c, d, e, f, g, h;
    kb_q4_bcast(a, sq, base + 0);
    kb_q4_bcast(b, sq, base + 1);
    kb_q4_bcast(c, sq, base + 2);
    kb_q4_bcast(d, sq, base + 3);
    fe_dbl(c, c);
    fe_add(h, a, b);
    fe_sub(e, h, d);
    fe_sub(g, a, b);
    fe_add(f, c, g);
    kb_q4_tail(p, e, f, g, h);
}
// p = p + q (sub = false) or p - q; `sub` is uniform over the quad
__device__ __forceinline__ void kb_q4_addsub(ge_p3& p, const ge_cached& q, bool sub)
{
    const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
    // role 0: (Y1 - X1) * (Y2 -+ X2)   1: (Y1 + X1) * (Y2 +- X2)   2: T1 * 2d T2   3: Z1 * Z2
    fe l, r, t, prod;
    fe_sub(l, p.Y, p.X);
    fe_add(t, p.Y, p.X);
    fe_cmov(l, t, (uint32_t)(role == 1));
    fe_cmov(l, p.T, (uint32_t)(role == 2));
    fe_cmov(l, p.Z, (uint32_t)(role == 3));
    r = sub ? q.YpX : q.YmX;
    t = sub ? q.YmX : q.YpX;
    fe_cmov(r, t, (uint32_t)(role == 1));
    fe_cmov(r, q.T2d, (uint32_t)(role == 2));
    fe_cmov(r, q.Z, (uint32_t)(role == 3));
    fe_mul(prod, l, r);
    fe a, b, c, d, e, f, g, h;
    kb_q4_bcast(a, prod, base + 0);
    kb_q4_bcast(b, prod, base + 1);
    kb_q4_bcast(c, prod, base + 2);
    kb_q4_bcast(d, prod, base + 3);
    fe_dbl(d, d);
    fe_sub(e, b, a);
    fe_add(h, b, a);
    if (sub) {
        fe_add(f, d, c);
        fe_sub(g, d, c);
    } else {
        fe_sub(f, d, c);
        fe_add(g, d, c);
    }
    kb_q4_tail(p, e, f, g, h);
}
// (the cached form of an operand costs one multiplication by 2d; doing it on one lane only would not shorten anything, so every lane does it)
__device__ __forceinline__ void kb_q4_conv_cell(ge_p3& v, const ge_p3& lower, bool has_self, const kb_naf& k)
{
    if (has_self) {
        ge_cached c;
        ge_to_cached(c, lower);
        kb_q4_addsub(v, c, false);
    } else {
        v = lower;
    }
    if (k.len <= 1) return;
    ge_cached vc;
    ge_to_cached(vc, v);
#pragma unroll 1
    for (int i = k.len - 2; i >= 0; i--) {
        const int d = k.d[i];
        kb_q4_dbl(v);
        if (d != 0) kb_q4_addsub(v, vc, d < 0);
    }
}
// k_fd_conv with four lanes per cell (same indexing; thread / 4 is the cell)
static __global__ void __launch_bounds__(KB_FD_CONV_THREADS) k_fd_conv_q4(size_t nd, size_t t, size_t h, size_t parts, size_t s, const uint32_t* dec, const uint32_t* src, uint32_t* dst)
{
    size_t idx = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    const size_t hl = kb_fd_part_len(t, h, parts - 1);
    const size_t sl = s + hl >= h ? s + hl - h : 0;
    const size_t cells = (parts - 1) * s + sl;
    const bool live = idx < nd * cells;
    if (!live) return;   // whole quads leave together (a quad is one cell)
    const size_t c = idx / nd, d = idx % nd;
    size_t q, k, sq, hq;
    if (c < (parts - 1) * s) {
        q = c % (parts - 1);
        k = s - c / (parts - 1);
        sq = s;
        hq = h;
    } else {
        q = parts - 1;
        k = sl - (c - (parts - 1) * s);
        sq = sl;
        hq = hl;
    }
    ge_p3 v, lower;
    if (k == 1) kb_load_p3_w128(lower, KB_FD_AT(dec, q * h + (hq - sq), d, nd));
    else kb_load_p3_w128(lower, KB_FD_AT(src, q * h + k - 1, d, nd));
    const bool has_self = k < sq;
    if (has_self) kb_load_p3_w128(v, KB_FD_AT(src, q * h + k, d, nd));
    else ge_identity(v);
    kb_naf kn;
    kb_naf_from(kn, (uint64_t)k);
    kb_q4_conv_cell(v, lower, has_self, kn);
    if ((threadIdx.x & 3) == 0) kb_store_p3_w128(KB_FD_AT(dst, q * h + k, d, nd), v);
}

// Stage C.  Block = one (dealer, block q); thread = order k.  All n steps in one launch: per step every lane turns its
// value into the operand form (1 M), hands it to the lane below (shuffle; the lowest lane of a warp through shared
// memory), adds what it received (8 M), and lane 0 records the value E_q(i + 1) into evals[(q * n + i) * nd + d].  An order
// k can only reach the value k steps later, so the orders above n - step are dead and their warps leave the loop.
// Neighbouring warps hand the operand over through a one-slot mailbox guarded by two NAMED barriers per pair (FULL: the
// upper warp arrives after writing, the lower warp waits; EMPTY: the lower warp arrives after reading, the upper warp
// waits before the next write), so a warp only ever waits for its neighbour and the six warps of a block run as a
// pipeline, up to one step apart per pair.  (A block-wide barrier per step was the largest stall of the first version of
// this kernel: ncu `barrier` 3.2 per issue.)
__device__ __forceinline__ void kb_bar_sync(unsigned id)
{
    asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory");
}
__device__ __forceinline__ void kb_bar_arrive(unsigned id)
{
    __threadfence_block();
    asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory");
}
template <int MAXH, int MINB>
static __global__ void __launch_bounds__(MAXH, MINB) k_fd_steps(size_t nd, size_t t, size_t h, size_t parts, size_t n, const uint32_t* dec, const uint32_t* diffs, uint32_t* evals)
{
    __shared__ uint4 xch_raw[(MAXH / 32) * 8];   // one mailbox of 32 words per warp: the operand of its lowest order
    uint32_t* xch = reinterpret_cast<uint32_t*>(xch_raw);
    // blocks of the same coefficient block are neighbours in the grid: the shorter last block (fewer live warps) comes
    // last and fills the tail of the launch
    const size_t q = blockIdx.x / nd, d = blockIdx.x % nd;
    const size_t hq = kb_fd_part_len(t, h, q);
    const unsigned k = threadIdx.x, lane = k & 31, warp = k >> 5;
    if (32u * warp >= hq) return;   // a warp without orders (the last coefficient block is shorter)
    const unsigned nlive = (unsigned)((hq + 31) / 32);
    ge_p3 p;
    ge_identity(p);
    if (k == 0) kb_load_p3_w128(p, KB_FD_AT(dec, q * h, d, nd));
    else if (k < hq) kb_load_p3_w128(p, KB_FD_AT(diffs, q * h + k, d, nd));
    const bool top = k + 1 >= hq;   // nothing above: the operand is the identity
    // barrier ids: pair (w, w + 1) uses FULL = 1 + 2 w and EMPTY = 2 + 2 w  (<= 14 for 8 warps; 0 is __syncthreads)
    const unsigned full_up = 1 + 2 * warp, empty_up = 2 + 2 * warp;            // as the consumer of the warp above
    const unsigned full_dn = 1 + 2 * (warp - 1), empty_dn = 2 + 2 * (warp - 1);  // as the producer for the warp below
    // the warp above produces for step i while it is live at step i
    if (warp + 1 < nlive && 32u * (warp + 1) <= n) kb_bar_arrive(empty_up);    // the mailbox starts empty
    for (size_t i = 0; i < n; i++) {
        const size_t reach = n - i;   // the orders <= reach can still matter
        if (32u * warp > reach) break;   // dead from here on (warp-uniform)
        ge_cached c;
        ge_to_cached(c, p);
        if (warp > 0) {
            kb_bar_sync(empty_dn);   // the warp below has read the previous operand
            if (lane == 0) kb_store_cached_w128(xch + 32 * warp, c);
            __syncwarp();
            kb_bar_arrive(full_dn);
        }
#pragma unroll
        for (int w = 0; w < 8; w++) {
            c.YpX.v[w] = __shfl_down_sync(0xffffffffu, c.YpX.v[w], 1);
            c.YmX.v[w] = __shfl_down_sync(0xffffffffu, c.YmX.v[w], 1);
            c.T2d.v[w] = __shfl_down_sync(0xffffffffu, c.T2d.v[w], 1);
            c.Z.v[w] = __shfl_down_sync(0xffffffffu, c.Z.v[w], 1);
        }
        // the warp above may be dead (its orders can no longer matter, so nor can this warp's top lane) or absent: the
        // operand then only has to be a valid point
        const bool above_live = warp + 1 < nlive && 32u * (warp + 1) <= reach;
        if (above_live) {
            kb_bar_sync(full_up);
            if (lane == 31) kb_load_cached_w128(c, xch + 32 * (warp + 1));
            __syncwarp();
            // the warp above only waits for this if it will produce again: at its next step it is live iff 32 (w+1) <= reach - 1
            if (32u * (warp + 1) + 1 <= reach) kb_bar_arrive(empty_up);
        } else if (lane == 31) {
            ge_cached_identity(c);
        }
        if (top) ge_cached_identity(c);
        ge_add<true>(p, p, c);
        if (k == 0) kb_store_p3_w128(evals + ((q * n + i) * nd + d) * 32, p);
    }
}

// Stage D: verdict[d * n + i] = [ P_d(i + 1) == share(d, i) * B ] and no undecodable commitment (vss/pedersen/vss.rs:899-912).
// Item idx = i * nd + d: the 32 lanes of a warp hold 32 dealers and ONE evaluation point, so the public multipliers
// x^(q h) mod 8L (pw) and with them every table index of the Straus loop are warp-uniform.  The share is secret: it only
// meets the constant-time select of the fixed-base comb staged in shared memory (ge_scalarmult_base<true>).
static __global__ void __launch_bounds__(KB_THREADS) k_fd_check(size_t nd, size_t n, size_t parts, const uint32_t* evals, const uint32_t* pw, const uint8_t* shares, const uint32_t* dealer_bad,
                                                                  const ge_precomp* table, uint8_t* verdict)
{
    extern __shared__ uint4 smem4[];
    ge_precomp* base = reinterpret_cast<ge_precomp*>(smem4);
    kb_stage(reinterpret_cast<uint32_t*>(base), reinterpret_cast<const uint32_t*>(table), 64 * 8 * 24);
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = idx < nd * n;   // the Straus loop holds block barriers: tail threads redo the last item
    if (!live) idx = nd * n - 1;
    const size_t i = idx / nd, d = idx % nd;
    const size_t slot = d * n + i;
    const int nt = (int)parts - 1;
    ge_cached tbl[8 * (KB_FD_MAX_PARTS - 1)];
    int8_t e[64 * (KB_FD_MAX_PARTS - 1)];
    uint32_t pw9[9 * (KB_FD_MAX_PARTS - 1)];
    for (int w = 0; w < 9 * nt; w++) pw9[w] = pw[i * 9 * nt + w];
    ge_p3 v;
    kb_fd_combine(v, nt, pw9, tbl, e, [&](int q, ge_p3& P) { kb_load_p3_w128(P, evals + (((size_t)q * n + i) * nd + d) * 32); });
    uint32_t s[8];
    int8_t es[64];
    kb_load32(s, shares, slot);
    sc_recode16(es, s);
    ge_p3 hb;
    ge_scalarmult_base<true>(hb, es, base);
    fe l, r, df;
    fe_mul(l, v.X, hb.Z);
    fe_mul(r, hb.X, v.Z);
    fe_sub(df, l, r);
    uint32_t same = fe_is_zero(df);
    fe_mul(l, v.Y, hb.Z);
    fe_mul(r, hb.Y, v.Z);
    fe_sub(df, l, r);
    same &= fe_is_zero(df);
    if (live) verdict[slot] = (uint8_t)(same & (dealer_bad[d] ? 0u : 1u));
}
// Stage D for SMALL shards: one item on four lanes.  With a few thousand (dealer, verifier) pairs — the 32 dealers of one
// rank of 8 in config 3 — the check kernel is a handful of warps that each run ~450 dependent point operations; the same
// quad-cooperative operations as in k_fd_conv_q4 shorten that chain 2.5x.  Every lane of a quad holds the whole item (its
// own copy of the tables in local memory); the share still only meets the constant-time scan of the comb in shared memory.
static __global__ void __launch_bounds__(KB_THREADS) k_fd_check_q4(size_t nd, size_t n, size_t parts, const uint32_t* evals, const uint32_t* pw, const uint8_t* shares, const uint32_t* dealer_bad,
                                                                     const ge_precomp* table, uint8_t* verdict)
{
    extern __shared__ uint4 smem4[];
    ge_precomp* base = reinterpret_cast<ge_precomp*>(smem4);
    kb_stage(reinterpret_cast<uint32_t*>(base), reinterpret_cast<const uint32_t*>(table), 64 * 8 * 24);
    size_t idx = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    const bool live = idx < nd * n;   // the loops hold block barriers: the quads past the end redo the last item
    if (!live) idx = nd * n - 1;
    const size_t i = idx / nd, d = idx % nd;
    const size_t slot = d * n + i;
    const int nt = (int)parts - 1;
    ge_cached tbl[8 * (KB_FD_MAX_PARTS - 1)];
    int8_t e[64 * (KB_FD_MAX_PARTS - 1)];
    ge_p3 P, W;
#pragma unroll 1
    for (int q = 0; q < nt; q++) {
        uint32_t pw9[9];
        for (int w = 0; w < 9; w++) pw9[w] = pw[i * 9 * nt + 9 * q + w];
        kb_load_p3_w128(P, evals + (((size_t)(q + 1) * n + i) * nd + d) * 32);
        if (pw9[8]) {
            fe_neg(P.X, P.X);
            fe_neg(P.T, P.T);
        }
        sc_recode16(e + 64 * q, pw9);
        // tbl[8 q + j] = (j + 1) P
        ge_p3 m = P;
        ge_to_cached(tbl[8 * q], P);
#pragma unroll 1
        for (int j = 1; j < 8; j++) {
            kb_q4_addsub(m, tbl[8 * q], false);
            ge_to_cached(tbl[8 * q + j], m);
        }
    }
    ge_identity(W);
    if (nt > 0) {
#pragma unroll 1
        for (int w = 63; w >= 0; w--) {
            KB_LOCKSTEP();
            if (w != 63) {
#pragma unroll 1
                for (int k = 0; k < 4; k++) kb_q4_dbl(W);
            }
#pragma unroll 1
            for (int q = 0; q < nt; q++) {
                ge_cached c;
                ge_select_cached<false>(c, tbl + 8 * q, e[64 * q + w]);   // public, warp-uniform digits
                kb_q4_addsub(W, c, false);
            }
        }
    }
    kb_load_p3_w128(P, evals + ((size_t)i * nd + d) * 32);
    ge_cached c0;
    ge_to_cached(c0, P);
    kb_q4_addsub(W, c0, false);
    // share * B through the constant-time comb: every lane scans the window itself, the addition runs on the quad
    uint32_t sw[8];
    int8_t es[64];
    kb_load32(sw, shares, slot);
    sc_recode16(es, sw);
    ge_p3 hb;
    ge_identity(hb);
#pragma unroll 1
    for (int w = 0; w < 64; w++) {
        ge_precomp pc;
        ge_select_precomp<true>(pc, base + 8 * w, es[w]);
        ge_cached c;
        c.YpX = pc.ypx;
        c.YmX = pc.ymx;
        c.T2d = pc.xy2d;
        fe_set(c.Z, 1);
        kb_q4_addsub(hb, c, false);
    }
    fe l, r, df;
    fe_mul(l, W.X, hb.Z);
    fe_mul(r, hb.X, W.Z);
    fe_sub(df, l, r);
    uint32_t same = fe_is_zero(df);
    fe_mul(l, W.Y, hb.Z);
    fe_mul(r, hb.Y, W.Z);
    fe_sub(df, l, r);
    same &= fe_is_zero(df);
    if (live && (threadIdx.x & 3) == 0) verdict[slot] = (uint8_t)(same & (dealer_bad[d] ? 0u : 1u));
}
#endif  // !KB_HOST_EMU
