// proto.cuh — kernels of the protocol-level entry points (capi_proto.cu): what the callers of the hot path do with
// its results, kept on the device so that nothing is compressed, copied out and decompressed between two steps.
//   session_id            share/vss/pedersen/vss.rs:1069-1090      k_points_decode_xyz / k_session_ids
//   find_pub              share/dkg/pedersen/dkg.rs:1109-1116      k_find_pub
//   rabin verify_deal     share/vss/rabin/vss.rs:889-900           k_rabin_finish
//   process_partial_sig   sign/dss/dss_sig.rs:263-273              k_dss_finish
//   recover_commit        share/poly.rs:566-603                    k_lagrange_coeffs / k_wmul / k_colsum
//   recover_pub_poly      share/poly.rs:607-635, :640-671          k_lagrange_basis / k_wmul / k_colsum
#pragma once
#include "kernels.cuh"
#include "msm.cuh"
#include "sha256.cuh"

// ---- encodings -> (X, Y, Z) for the batch compressor; bad[i] = 1 (and the identity) where the input does not decode
static __global__ void __launch_bounds__(KB_THREADS) k_points_decode_xyz(size_t n, const uint8_t* in, uint32_t* xyz, uint8_t* bad)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[8];
    kb_load32(w, in, i);
    ge_p3 p;
    const uint32_t ok = ge_decompress(p, w);
    if (!ok) ge_identity(p);
    kb_store_xyz(xyz, i, p);
    bad[i] = (uint8_t)(ok ^ 1u);
}

// ---- session_id: sid_d = SHA-256(dealer_d || verifier_0 .. verifier_(n-1) || commit_(d,0) .. commit_(d,t-1) || t as u32 LE)
// over CANONICAL encodings (marshal_to re-encodes the point).  One thread per dealer.
// The three arrays are consecutive in ONE buffer of encodings (dealers, verifiers, commits), `bad` runs parallel to it:
// status[d] = 1 if a point that went into sid_d did not decode (the reference could not hold such a point).
static __global__ void __launch_bounds__(32) k_session_ids(size_t nd, size_t n, size_t t, const uint8_t* dealers, const uint8_t* verifiers, const uint8_t* commits, const uint8_t* bad, uint8_t* out, uint8_t* status)
{
    const size_t d = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= nd) return;
    const uint8_t *bad_v = bad + nd, *bad_c = bad + nd + n;
    kb_sha256 s;
    sha256_init(s);
    uint32_t w[8];
    uint32_t anybad = bad[d];
    kb_load32(w, dealers, d);
    sha256_rec32(s, w);
    for (size_t i = 0; i < n; i++) {
        kb_load32(w, verifiers, i);
        sha256_rec32(s, w);
        anybad |= bad_v[i];
    }
    for (size_t j = 0; j < t; j++) {
        kb_load32(w, commits, d * t + j);
        sha256_rec32(s, w);
        anybad |= bad_c[d * t + j];
    }
    const uint32_t tw = (uint32_t)t;
    sha256_words(s, &tw, 1);
    sha256_final(s, w);
    kb_store32(out, d, w);
    status[d] = (uint8_t)(anybad != 0);
}

// ---- find_pub: index of the first list entry whose canonical encoding equals the query's, -1 if none, -2 if the query
// does not decode (qbad).  Entries that do not decode (lbad) never match.
static __global__ void __launch_bounds__(KB_THREADS) k_find_pub(size_t nlist, const uint8_t* list, const uint8_t* lbad, size_t m, const uint8_t* queries, const uint8_t* qbad, int32_t* out)
{
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    if (qbad[k]) {
        out[k] = -2;
        return;
    }
    uint32_t q[8], w[8];
    kb_load32(q, queries, k);
    int32_t found = -1;
    for (size_t i = 0; i < nlist && found < 0; i++) {
        kb_load32(w, list, i);
        uint32_t diff = 0;
#pragma unroll
        for (int c = 0; c < 8; c++) diff |= w[c] ^ q[c];
        if (diff == 0 && !lbad[i]) found = (int32_t)i;
    }
    out[k] = found;
}

// (X : Y : Z) -> extended (X Z : Y Z : Z^2 : X Y), the same point with a consistent T
__device__ __forceinline__ void kb_load_xyz_ext(ge_p3& p, const uint32_t* xyz, size_t i)
{
    fe x, y, z;
    kb_load_xyz(x, y, z, xyz, i);
    fe_mul(p.X, x, z);
    fe_mul(p.Y, y, z);
    fe_sq(p.Z, z);
    fe_mul(p.T, x, y);
}
__device__ __forceinline__ uint32_t kb_proj_equal(const ge_p3& a, const ge_p3& b)
{
    fe l, r, df;
    fe_mul(l, a.X, b.Z);
    fe_mul(r, b.X, a.Z);
    fe_sub(df, l, r);
    uint32_t same = fe_is_zero(df);
    fe_mul(l, a.Y, b.Z);
    fe_mul(r, b.Y, a.Z);
    fe_sub(df, l, r);
    return same & fe_is_zero(df);
}

// ---- rabin verify_deal: verdict[k] = [ f_k * G + g_k * H == eval_k ]  (share/vss/rabin/vss.rs:889-900).
// eval = PubPoly::eval results left by k_poly_eval as (X, Y, Z); both shares are secret: the fixed base through the
// constant-time comb staged in shared memory, H through the constant-time window select of ge_scalarmult<true>.
static __global__ void __launch_bounds__(KB_THREADS) k_rabin_finish(size_t m, const uint32_t* xyz, const uint8_t* bad, const uint8_t* f_shares, const uint8_t* g_shares, const uint8_t* h_point,
                                                                      const ge_precomp* table, uint8_t* verdict)
{
    extern __shared__ uint4 smem4[];
    ge_precomp* base = reinterpret_cast<ge_precomp*>(smem4);
    kb_stage(reinterpret_cast<uint32_t*>(base), reinterpret_cast<const uint32_t*>(table), 64 * 8 * 24);
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = k < m;   // ge_scalarmult holds block barriers: tail threads redo the last item
    if (!live) k = m - 1;
    uint32_t s[8], hw[8];
    int8_t e[64];
    ge_cached tbl[8];
    ge_p3 H, gh, fb, v;
    kb_load32(hw, h_point, 0);
    const uint32_t h_ok = ge_decompress(H, hw);
    kb_load32(s, g_shares, k);
    sc_recode16(e, s);
    ge_build_table8(tbl, H);
    ge_scalarmult<true>(gh, e, tbl);
    kb_load32(s, f_shares, k);
    sc_recode16(e, s);
    ge_scalarmult_base<true>(fb, e, base);
    ge_cached c;
    ge_to_cached(c, gh);
    ge_add<true>(fb, fb, c);
    kb_load_xyz(v.X, v.Y, v.Z, xyz, k);
    const uint32_t same = kb_proj_equal(v, fb);
    if (live) verdict[k] = (uint8_t)(same & h_ok & (bad[k] ? 0u : 1u));
}

// ---- DSS partial signatures: verdict[k] = [ partial_k * B == rand_eval_k + hash * long_eval_k ]  (sign/dss/dss_sig.rs:263-273).
// xyz holds the 2 m evaluations left by k_poly_eval: [0, m) of the random polynomial, [m, 2m) of the long-term one.
// Everything here is public (a partial signature is a broadcast message).
static __global__ void __launch_bounds__(KB_THREADS) k_dss_finish(size_t m, const uint32_t* xyz, const uint8_t* bad, const uint8_t* hash32, const uint8_t* partials, const ge_precomp* comb, uint8_t* verdict)
{
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = k < m;
    if (!live) k = m - 1;
    uint32_t s[8];
    int8_t e[64];
    ge_cached tbl[8];
    ge_p3 vl, right, vr, left;
    kb_load32(s, hash32, 0);
    sc_recode16(e, s);
    kb_load_xyz_ext(vl, xyz, m + k);
    ge_build_table8(tbl, vl);
    ge_scalarmult<false>(right, e, tbl);
    kb_load_xyz_ext(vr, xyz, k);
    ge_cached c;
    ge_to_cached(c, vr);
    ge_add<true>(right, right, c);
    kb_load32(s, partials, k);
    ge_scalarmult_base_comb(left, s, comb);
    const uint32_t same = kb_proj_equal(left, right);
    if (live) verdict[k] = (uint8_t)(same & ((bad[k] | bad[m + k]) ? 0u : 1u));
}

// ---- Lagrange coefficients at 0 on the nodes x_i = idx_i + 1 (share/poly.rs:583-597):
//   lam_i = prod_{j != i} x_j / prod_{j != i} (x_j - x_i)  mod L
static __global__ void __launch_bounds__(KB_THREADS) k_lagrange_coeffs(size_t k, const uint32_t* idx, uint8_t* lam)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t num[8] = {1, 0, 0, 0, 0, 0, 0, 0}, den[8] = {1, 0, 0, 0, 0, 0, 0, 0};
    uint32_t xi[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const uint64_t xiv = (uint64_t)idx[i] + 1;
    xi[0] = (uint32_t)xiv;
    xi[1] = (uint32_t)(xiv >> 32);
    for (size_t j = 0; j < k; j++) {
        if (j == i) continue;
        uint32_t xj[8] = {0, 0, 0, 0, 0, 0, 0, 0}, df[8];
        const uint64_t xjv = (uint64_t)idx[j] + 1;
        xj[0] = (uint32_t)xjv;
        xj[1] = (uint32_t)(xjv >> 32);
        sc_muladd(num, num, xj, zero);
        sc_sub_mod(df, xj, xi);
        sc_muladd(den, den, df, zero);
    }
    uint32_t inv[8], r[8];
    sc_invert(inv, den);
    sc_muladd(r, num, inv, zero);
    kb_store32(lam, i, r);
}

// ---- Lagrange BASIS polynomials on the nodes x_j = idx_j + 1 (lagrange_basis, share/poly.rs:640-671):
//   basis_j(x) = prod_{m != j} (x - x_m) / prod_{m != j} (x_j - x_m);   out[c * k + j] = coefficient c of basis_j.
// One block of k threads (k <= 1024): the master polynomial M(x) = prod_m (x - x_m) is built in shared memory, one
// root per step; thread j then divides it by (x - x_j) synthetically and scales by 1 / M'(x_j).
static __global__ void __launch_bounds__(1024) k_lagrange_basis(size_t k, const uint32_t* idx, uint8_t* out)
{
    extern __shared__ uint4 smem4[];
    uint32_t* mc = reinterpret_cast<uint32_t*>(smem4);   // (k + 1) x 8 words: coefficients of M, low order first
    const size_t j = threadIdx.x;                         // blockDim.x = k + 1: thread j owns coefficient j
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const uint32_t lm1[8] = {0x5cf5d3ecu, 0x5812631au, 0xa2f79cd6u, 0x14def9deu, 0u, 0u, 0u, 0x10000000u};   // L - 1 = -1
    for (int w = 0; w < 8; w++) mc[8 * j + w] = (j == 0 && w == 0) ? 1u : 0u;   // M = 1
    __syncthreads();
    for (size_t m = 0; m < k; m++) {
        // M <- M * (x - x_m):  c'_i = c_(i-1) - x_m c_i
        uint32_t xm[8] = {0, 0, 0, 0, 0, 0, 0, 0}, nx[8], ci[8], cm[8], r[8];
        const uint64_t xv = (uint64_t)idx[m] + 1;
        xm[0] = (uint32_t)xv;
        xm[1] = (uint32_t)(xv >> 32);
        sc_muladd(nx, lm1, xm, zero);   // -x_m
        for (int w = 0; w < 8; w++) {
            ci[w] = mc[8 * j + w];                          // zero above the current degree
            cm[w] = (j >= 1) ? mc[8 * (j - 1) + w] : 0u;
        }
        sc_muladd(r, nx, ci, cm);
        __syncthreads();
        for (int w = 0; w < 8; w++) mc[8 * j + w] = r[w];
        __syncthreads();
    }
    if (j >= k) return;
    uint32_t xj[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const uint64_t xjv = (uint64_t)idx[j] + 1;
    xj[0] = (uint32_t)xjv;
    xj[1] = (uint32_t)(xjv >> 32);
    // 1 / prod_{m != j} (x_j - x_m)
    uint32_t den[8] = {1, 0, 0, 0, 0, 0, 0, 0};
    for (size_t m = 0; m < k; m++) {
        if (m == j) continue;
        uint32_t xm[8] = {0, 0, 0, 0, 0, 0, 0, 0}, df[8];
        const uint64_t xv = (uint64_t)idx[m] + 1;
        xm[0] = (uint32_t)xv;
        xm[1] = (uint32_t)(xv >> 32);
        sc_sub_mod(df, xj, xm);
        sc_muladd(den, den, df, zero);
    }
    uint32_t acc[8];
    sc_invert(acc, den);
    // synthetic division by (x - x_j): b_(k-1) = c_k, b_(i-1) = c_i + x_j b_i
    uint32_t b[8];
    for (int w = 0; w < 8; w++) b[w] = mc[8 * k + w];
    for (size_t i = k; i-- > 0;) {
        uint32_t o[8];
        sc_muladd(o, b, acc, zero);
        kb_store32(out, i * k + j, o);   // coefficient i of basis_j
        if (i > 0) {
            uint32_t ci[8];
            for (int w = 0; w < 8; w++) ci[w] = mc[8 * i + w];
            sc_muladd(b, xj, b, ci);
        }
    }
}

// ---- out128[c * k + i] = s * P as an extended point, for the weighted column sums of recover_commit / recover_pub_poly.
// scalars: k x 32 bytes shared by all columns (s_per_col = 0) or ncols x k (s_per_col = 1); points likewise (32-byte
// encodings).  Public data: indexed table lookups; the window schedule is the same for every thread.
// bad[c * k + i] = 1 where the point does not decode.
static __global__ void __launch_bounds__(KB_THREADS) k_wmul(size_t ncols, size_t k, const uint8_t* scalars, int s_per_col, const uint8_t* points, int p_per_col, uint32_t* out128, uint8_t* bad)
{
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = idx < ncols * k;
    if (!live) idx = ncols * k - 1;
    // lanes = columns for a shared scalar (warp-uniform digits), = rows otherwise
    const size_t c = s_per_col ? idx / k : idx % ncols, i = s_per_col ? idx % k : idx / ncols;
    uint32_t s[8], w[8];
    int8_t e[64];
    ge_cached tbl[8];
    kb_load32(s, scalars, s_per_col ? c * k + i : i);
    kb_load32(w, points, p_per_col ? c * k + i : i);
    ge_p3 p, h;
    const uint32_t ok = ge_decompress(p, w);
    sc_recode16(e, s);
    ge_build_table8(tbl, p);
    ge_scalarmult<false>(h, e, tbl);
    if (!ok) ge_identity(h);
    if (!live) return;
    kb_store_p3_w32(out128 + 32 * (c * k + i), h);
    bad[c * k + i] = (uint8_t)(ok ^ 1u);
}
// xyz[c] = sum_i in128[c * k + i]; status[c] = 1 if any of them was flagged.  One warp per column.
static __global__ void __launch_bounds__(KB_THREADS) k_colsum(size_t ncols, size_t k, const uint32_t* in128, const uint8_t* bad, uint32_t* xyz, uint8_t* status)
{
    const uint32_t lane = threadIdx.x & 31;
    const size_t c = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (c >= ncols) return;
    ge_p3 s;
    ge_identity(s);
    uint32_t anybad = 0;
    for (size_t i = lane; i < k; i += 32) {
        ge_p3 p;
        kb_load_p3_w32(p, in128 + 32 * (c * k + i));
        ge_cached pc;
        ge_to_cached(pc, p);
        ge_add<true>(s, s, pc);
        anybad |= bad[c * k + i];
    }
    kb_warp_sum_point(s);
    anybad = __any_sync(0xffffffffu, anybad != 0);
    if (lane == 0) {
        if (anybad) ge_identity(s);
        kb_store_xyz(xyz, c, s);
        status[c] = (uint8_t)anybad;
    }
}
// out[c * k + i] = in[i * ncols + c]: 32-byte records, for resharing_key's "take all i-th coefficients" (dkg.rs:1003-1016)
static __global__ void __launch_bounds__(256) k_transpose32(size_t rows, size_t cols, const uint8_t* in, uint8_t* out)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * cols) return;
    const size_t r = idx / cols, c = idx % cols;
    uint32_t w[8];
    kb_load32(w, in, idx);
    kb_store32(out, c * rows + r, w);
}
