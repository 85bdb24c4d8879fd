// kernels.cuh — __global__ entry points.  One thread owns one item; the math lives in
// ops.cuh / poly.cuh.  Data crosses HBM in the reference's wire encodings (32-byte points
// and scalars), loaded and stored as 128-bit vectors.
#pragma once
#include <cuda_runtime.h>
#include "ops.cuh"
#include "poly.cuh"

#define KB_THREADS 128

// 32-byte record i of a 16-byte-aligned array -> 8 LE words (two 128-bit loads)
__device__ __forceinline__ void kb_load32(uint32_t* w, const uint8_t* base, size_t i)
{
    const uint4* p = reinterpret_cast<const uint4*>(base + 32 * i);
    uint4 a = __ldg(p), b = __ldg(p + 1);
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
    w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
}
__device__ __forceinline__ void kb_store32(uint8_t* base, size_t i, const uint32_t* w)
{
    uint4* p = reinterpret_cast<uint4*>(base + 32 * i);
    p[0] = make_uint4(w[0], w[1], w[2], w[3]);
    p[1] = make_uint4(w[4], w[5], w[6], w[7]);
}
// streaming (evict-first) variants for data that crosses HBM exactly once — the records between the two verify
// launches — so that it does not push the per-thread tables out of L2
__device__ __forceinline__ void kb_load_fe_cs(fe& f, const uint32_t* p)
{
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = __ldcs(q), b = __ldcs(q + 1);
    f.v[0] = a.x; f.v[1] = a.y; f.v[2] = a.z; f.v[3] = a.w;
    f.v[4] = b.x; f.v[5] = b.y; f.v[6] = b.z; f.v[7] = b.w;
}
__device__ __forceinline__ void kb_store_fe_cs(uint32_t* p, const fe& f)
{
    uint4* q = reinterpret_cast<uint4*>(p);
    __stcs(q, make_uint4(f.v[0], f.v[1], f.v[2], f.v[3]));
    __stcs(q + 1, make_uint4(f.v[4], f.v[5], f.v[6], f.v[7]));
}
// cooperative copy of `words` 32-bit words from global to shared
__device__ __forceinline__ void kb_stage(uint32_t* dst, const uint32_t* src, int words)
{
    const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    for (int i = threadIdx.x; i < words / 4; i += blockDim.x) d[i] = __ldg(s + i);
    __syncthreads();
}

// Kernel groups: a translation unit defines KB_K_POINT / KB_K_SIGN / KB_K_POLY / KB_K_MSM / KB_K_KEYSET for the non-template kernels it
// launches (nvcc compiles every __global__ function it sees, used or not).
#if defined(KB_K_POINT)
// ---- base-point table: table[w*8 + j] = (j+1) * 16^w * B, w = 0..63 (replaces constants.rs:89 BASE)
static __global__ void k_base_init(ge_precomp* table)
{
    const int w = threadIdx.x;
    if (w >= 64) return;
    ge_p3 pos;
    const fe bx = KB_FE_BX, by = KB_FE_BY, bt = KB_FE_BT;
    pos.X = bx; pos.Y = by; pos.T = bt;
    fe_set(pos.Z, 1);
    for (int k = 0; k < 4 * w; k++) ge_dbl<true>(pos, pos);
    kb_base_window(table + 8 * w, pos);
}

// base128[j] = (j+1) * B, j = 0..127: the radix-256 fixed-base table of the full-length verifiers
static __global__ void k_base128_init(ge_precomp* table)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    ge_p3 pos;
    const fe bx = KB_FE_BX, by = KB_FE_BY, bt = KB_FE_BT;
    pos.X = bx; pos.Y = by; pos.T = bt;
    fe_set(pos.Z, 1);
    kb_base_window(table, pos, 128);
}
// comb[p][j] = (j+1) * 2^(KB_COMB_BITS p) * B: the fixed-base comb of the half-size-scalar verifiers (ops.cuh)
static __global__ void __launch_bounds__(KB_THREADS) k_comb_init(ge_precomp* comb, const ge_precomp* base_table)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= KB_COMB_POS * KB_COMB_HALF) return;
    ge_precomp e;
    kb_comb_entry(e, k / KB_COMB_HALF, k % KB_COMB_HALF, base_table);
    comb[k] = e;
}

#endif  // KB_K_POINT
// ---- shared tail of every point-producing kernel: Montgomery's trick over KB_INV_K results -----
// Stage-1 kernels leave (X, Y, Z) in `xyz` (24 words per item).  One thread then owns KB_INV_K
// consecutive items, multiplies their Z's together, inverts ONCE (fe_invert, 254S + 11M) and
// unwinds: 3 multiplications per item instead of an inversion each (write_bytes, ge.rs:112-122,
// pays one per point).  Items whose stage 1 failed carry Z = 1.
#define KB_INV_K 8
__device__ __forceinline__ void kb_store_xyz(uint32_t* xyz, size_t i, const ge_p3& p)
{
    uint32_t* o = xyz + 24 * i;
    kb_store_fe(o, p.X);
    kb_store_fe(o + 8, p.Y);
    kb_store_fe(o + 16, p.Z);
}
__device__ __forceinline__ void kb_load_xyz_xy(fe& x, fe& y, const uint32_t* xyz, size_t i)
{
    kb_load_fe(x, xyz + 24 * i);
    kb_load_fe(y, xyz + 24 * i + 8);
}
__device__ __forceinline__ void kb_load_xyz_z(fe& z, const uint32_t* xyz, size_t i) { kb_load_fe(z, xyz + 24 * i + 16); }
__device__ __forceinline__ void kb_load_xyz(fe& x, fe& y, fe& z, const uint32_t* xyz, size_t i)
{
    kb_load_xyz_xy(x, y, xyz, i);
    kb_load_xyz_z(z, xyz, i);
}
// calls emit(i, enc[8]) for every item of this thread's group, enc = canonical encoding
template <typename F>
__device__ __forceinline__ void kb_batch_compress(size_t n, const uint32_t* xyz, F emit)
{
    const size_t base = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * KB_INV_K;
    if (base >= n) return;
    const int cnt = (n - base < KB_INV_K) ? (int)(n - base) : KB_INV_K;
    fe pref[KB_INV_K];
    fe acc, z;
    kb_load_xyz_z(acc, xyz, base);
    pref[0] = acc;
#pragma unroll 1
    for (int k = 1; k < cnt; k++) {
        kb_load_xyz_z(z, xyz, base + k);
        fe_mul(acc, acc, z);
        pref[k] = acc;
    }
    fe inv;
    fe_invert(inv, acc);
#pragma unroll 1
    for (int k = cnt - 1; k >= 0; k--) {
        fe zinv;
        if (k > 0) {
            fe_mul(zinv, inv, pref[k - 1]);
            kb_load_xyz_z(z, xyz, base + k);
            fe_mul(inv, inv, z);
        } else {
            zinv = inv;
        }
        ge_p3 p;
        kb_load_xyz_xy(p.X, p.Y, xyz, base + k);
        uint32_t enc[8];
        ge_compress_with_zinv(enc, p, zinv);
        emit(base + k, enc);
    }
}
// out[i] = encoding of item i; zeroed where bad[i] != 0
static __global__ void __launch_bounds__(KB_THREADS) k_compress_batch(size_t n, const uint32_t* xyz, const uint8_t* bad, uint8_t* out)
{
    kb_batch_compress(n, xyz, [&](size_t i, uint32_t* enc) {
        if (bad && bad[i]) {
#pragma unroll
            for (int q = 0; q < 8; q++) enc[q] = 0;
        }
        kb_store32(out, i, enc);
    });
}

// ---- serde wire format of the reference: raw ExtendedGroupElement limbs -> (X, Y, Z) for the batch
// compressor.  Z = 0 (e.g. Point::default(), all-zero limbs) encodes as 32 zero bytes in the reference
// (fe_invert(0) = 0, ge.rs:112-122): flagged in zero_out and replaced by Z = 1 so that the shared inversion
// of its group stays valid.
static __global__ void __launch_bounds__(KB_THREADS) k_points_from_limbs(size_t n, const int32_t* limbs, uint32_t* xyz, uint8_t* zero_out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t l[30];
    const int4* src = reinterpret_cast<const int4*>(limbs + 40 * i);   // 160-byte records: 16-byte aligned
#pragma unroll
    for (int k = 0; k < 7; k++) {
        const int4 q = __ldg(src + k);
        l[4 * k] = q.x; l[4 * k + 1] = q.y;
        if (4 * k + 2 < 30) { l[4 * k + 2] = q.z; l[4 * k + 3] = q.w; }
    }
    {
        const int4 q = __ldg(src + 7);
        l[28] = q.x; l[29] = q.y;
    }
    ge_p3 p;
    fe_from_ref10(p.X, l);
    fe_from_ref10(p.Y, l + 10);
    fe_from_ref10(p.Z, l + 20);
    const uint32_t z0 = fe_is_zero(p.Z);
    if (z0) ge_identity(p);
    kb_store_xyz(xyz, i, p);
    zero_out[i] = (uint8_t)z0;
}

#if defined(KB_K_POINT)
// ---- Point::mul(s, None): out[i] = compress(s_i * B)   (point.rs:207, ge.rs:442)
// `split` (1, 2 or 4) adjacent lanes share one scalar: each walks 64/split of the comb windows and the partial
// points are added with a shuffle butterfly.  The comb has no doublings, so the windows are independent; small
// batches (config 1 is 2^16 scalars, a fraction of what 148 SMs hold) then occupy 2-4x more lanes.
__device__ __forceinline__ void kb_shfl_xor_point(ge_p3& q, const ge_p3& p, int off)
{
#pragma unroll
    for (int k = 0; k < 8; k++) {
        q.X.v[k] = __shfl_xor_sync(0xffffffffu, p.X.v[k], off);
        q.Y.v[k] = __shfl_xor_sync(0xffffffffu, p.Y.v[k], off);
        q.Z.v[k] = __shfl_xor_sync(0xffffffffu, p.Z.v[k], off);
        q.T.v[k] = __shfl_xor_sync(0xffffffffu, p.T.v[k], off);
    }
}
template <bool CT>
static __global__ void __launch_bounds__(KB_THREADS) k_mul_base(size_t n, const uint8_t* scalars, uint32_t* xyz, const ge_precomp* table, int split)
{
    extern __shared__ uint4 smem4[];
    ge_precomp* base = reinterpret_cast<ge_precomp*>(smem4);
    kb_stage(reinterpret_cast<uint32_t*>(base), reinterpret_cast<const uint32_t*>(table), 64 * 8 * 24);
    const size_t gtid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t i = gtid / split;
    const int part = (int)(gtid % split);
    const bool live = i < n;   // whole warps take part in the shuffles: tail lanes redo the last scalar
    if (!live) i = n - 1;
    uint32_t s[8];
    int8_t e[64];
    kb_load32(s, scalars, i);
    sc_recode16(e, s);
    ge_p3 h;
    const int per = 64 / split;
    ge_scalarmult_base<CT>(h, e, base, part * per, (part + 1) * per);
    for (int off = 1; off < split; off <<= 1) {
        ge_p3 q;
        kb_shfl_xor_point(q, h, off);
        ge_cached qc;
        ge_to_cached(qc, q);
        ge_add<true>(h, h, qc);
    }
    if (live && part == 0) kb_store_xyz(xyz, i, h);
}

// public scalars (KB_FLAG_VARTIME): the shared comb, KB_COMB_POS (15) mixed additions per scalar, nothing staged in shared memory
static __global__ void __launch_bounds__(KB_THREADS) k_mul_base_comb(size_t n, const uint8_t* scalars, uint32_t* xyz, const ge_precomp* comb)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t s[8];
    kb_load32(s, scalars, i);
    ge_p3 h;
    ge_scalarmult_base_comb(h, s, comb);
    kb_store_xyz(xyz, i, h);
}

// ---- Point::mul(s, Some(p)): out[i] = compress(s_i * P_i)   (point.rs:207, ge.rs:508)
template <bool CT>
static __global__ void __launch_bounds__(KB_THREADS) k_mul(size_t n, const uint8_t* scalars, const uint8_t* points, int shared_point, uint32_t* xyz, uint8_t* status)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n;   // ge_scalarmult holds block barriers: tail threads redo the last item
    if (!live) i = n - 1;
    uint32_t s[8], w[8];
    int8_t e[64];
    ge_cached tbl[8];
    kb_load32(s, scalars, i);
    kb_load32(w, points, shared_point ? 0 : i);
    ge_p3 p, h;
    const uint32_t ok = ge_decompress(p, w);
    sc_recode16(e, s);
    ge_build_table8(tbl, p);
    ge_scalarmult<CT>(h, e, tbl);
    if (!ok) ge_identity(h);
    if (!live) return;
    kb_store_xyz(xyz, i, h);
    if (status) status[i] = (uint8_t)(ok ^ 1u);
}

// ---- Point::unmarshal_binary + marshal_binary   (ge.rs:124, :112)
static __global__ void __launch_bounds__(KB_THREADS) k_recode(size_t n, const uint8_t* in, uint8_t* out, uint8_t* status)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[8], o[8];
    kb_load32(w, in, i);
    ge_p3 p;
    const uint32_t ok = ge_decompress(p, w);
    ge_compress(o, p);
    if (!ok) {
#pragma unroll
        for (int k = 0; k < 8; k++) o[k] = 0;
    }
    kb_store32(out, i, o);
    if (status) status[i] = (uint8_t)(ok ^ 1u);
}

// ---- Point::add / Point::sub   (point.rs:179, :190)
static __global__ void __launch_bounds__(KB_THREADS) k_point_add(size_t n, const uint8_t* pa, const uint8_t* pb, uint8_t* out, uint8_t* status, int subtract)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[8], o[8];
    ge_p3 p, q, r;
    kb_load32(w, pa, i);
    uint32_t ok = ge_decompress(p, w);
    kb_load32(w, pb, i);
    ok &= ge_decompress(q, w);
    ge_cached c;
    ge_to_cached(c, q);
    ge_cached_cneg(c, (uint32_t)(subtract != 0));
    ge_add<false>(r, p, c);
    ge_compress(o, r);
    if (!ok) {
#pragma unroll
        for (int k = 0; k < 8; k++) o[k] = 0;
    }
    kb_store32(out, i, o);
    if (status) status[i] = (uint8_t)(ok ^ 1u);
}

// ---- the uncompressed, device-friendly form for chaining: X, Y, Z, T as 4 x 8 little-endian words (128 bytes per
// point, the form kb_msm's partial sums use).  ExtendedGroupElement::set_bytes / write_bytes (ge.rs:124, :112).
static __global__ void __launch_bounds__(KB_THREADS) k_point_decompress(size_t n, const uint8_t* in, uint32_t* out128, uint8_t* status)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[8];
    kb_load32(w, in, i);
    ge_p3 p;
    const uint32_t ok = ge_decompress(p, w);
    if (!ok) ge_identity(p);
    kb_store_p3_w128(out128 + 32 * i, p);
    if (status) status[i] = (uint8_t)(ok ^ 1u);
}
// 128-byte form -> (X, Y, Z) for the batch compressor; Z = 0 encodes as 32 zero bytes (fe_invert(0) = 0, ge.rs:112-122)
static __global__ void __launch_bounds__(KB_THREADS) k_points_from_raw(size_t n, const uint32_t* in128, uint32_t* xyz, uint8_t* zero_out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ge_p3 p;
    kb_load_p3_xy_w128(p.X, p.Y, in128 + 32 * i);
    kb_load_p3_z_w128(p.Z, in128 + 32 * i);
    const uint32_t z0 = fe_is_zero(p.Z);
    if (z0) ge_identity(p);
    kb_store_xyz(xyz, i, p);
    zero_out[i] = (uint8_t)z0;
}
// ---- Point::eq (point.rs:227-241): equality of the canonical encodings of two decoded points; bit 1 of the
// result flags an operand that does not decode (the reference cannot even construct such a Point)
static __global__ void __launch_bounds__(KB_THREADS) k_point_eq(size_t n, const uint8_t* pa, const uint8_t* pb, uint8_t* out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[8];
    ge_p3 p, q;
    kb_load32(w, pa, i);
    uint32_t ok = ge_decompress(p, w);
    kb_load32(w, pb, i);
    ok &= ge_decompress(q, w);
    fe d;   // both have Z = 1
    fe_sub(d, p.X, q.X);
    uint32_t same = fe_is_zero(d);
    fe_sub(d, p.Y, q.Y);
    same &= fe_is_zero(d);
    out[i] = (uint8_t)((same & ok) | ((ok ^ 1u) << 1));
}

// ---- Point::is_canonical / has_small_order / decodes   (point.rs:322, :286; ge.rs:124)
static __global__ void __launch_bounds__(KB_THREADS) k_point_check(size_t n, const uint8_t* in, uint8_t* flags)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[8], o[8];
    kb_load32(w, in, i);
    ge_p3 p;
    const uint32_t ok = ge_decompress(p, w);
    uint32_t small = 0;
    if (ok) {
        ge_compress(o, p);  // has_small_order works on the re-encoding
        small = pt_is_small_order_bytes(o);
    }
    flags[i] = (uint8_t)(pt_is_canonical(w) | (small << 1) | (ok << 2));
}

// ---- scalars   (scalar.rs:175, :279)
static __global__ void __launch_bounds__(KB_THREADS) k_sc_reduce64(size_t n, const uint8_t* in, uint8_t* out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t x[16], r[8];
    kb_load32(x, in, 2 * i);
    kb_load32(x + 8, in, 2 * i + 1);
    sc_reduce512(r, x);
    kb_store32(out, i, r);
}
static __global__ void __launch_bounds__(KB_THREADS) k_sc_muladd(size_t n, const uint8_t* a, const uint8_t* b, const uint8_t* c, uint8_t* out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t A[8], B[8], C[8], r[8];
    kb_load32(A, a, i);
    kb_load32(B, b, i);
    kb_load32(C, c, i);
    sc_muladd(r, A, B, C);
    kb_store32(out, i, r);
}
// Scalar::inv (scalar.rs:192)
static __global__ void __launch_bounds__(KB_THREADS) k_sc_invert(size_t n, const uint8_t* a, uint8_t* out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t A[8], r[8];
    kb_load32(A, a, i);
    sc_invert(r, A);
    kb_store32(out, i, r);
}
// h_i = SHA-512(R_i || A_i || M_i) mod L   (eddsa_sig.rs:195-200)
static __global__ void __launch_bounds__(KB_THREADS) k_challenge(size_t n, const uint8_t* r32, const uint8_t* a32, const uint8_t* msg, const uint64_t* msg_off, uint8_t* out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t rw[8], aw[8], d[16], h[8];
    kb_load32(rw, r32, i);
    kb_load32(aw, a32, i);
    const uint64_t lo = msg_off[i], hi = msg_off[i + 1];
    sha512_ram(d, rw, aw, msg + lo, hi - lo);
    sc_reduce512(h, d);
    kb_store32(out, i, h);
}

#endif  // KB_K_POINT
#if defined(KB_K_SIGN)
// ---- EdDSA::sign (sign/eddsa/eddsa_sig.rs:120-152) with the key derivation of
// Curve::new_key_and_seed_with_input (group/edwards25519/curve.rs:74-87), three launches:
//   k_sign_stage1   (a, prefix) = clamp(SHA-512(seed)); r = SHA-512(prefix || M) mod L; r*B and a*B (constant-time comb)
//   k_compress_batch on the 2n points  ->  R and A encodings
//   k_sign_finish   h = SHA-512(R || A || M) mod L; s = (r + h*a) mod L; sig = R || s
// The secret scalars a and r only ever meet the constant-time select (no secret-dependent address or branch).
static __global__ void __launch_bounds__(KB_THREADS) k_sign_stage1(size_t n, const uint8_t* seeds, const uint8_t* msg, const uint64_t* msg_off, uint32_t* xyz, uint8_t* a_out, uint8_t* r_out,
                                                            const ge_precomp* table)
{
    extern __shared__ uint4 smem4[];
    ge_precomp* base = reinterpret_cast<ge_precomp*>(smem4);
    kb_stage(reinterpret_cast<uint32_t*>(base), reinterpret_cast<const uint32_t*>(table), 64 * 8 * 24);
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t seed[8], d[16], a[8], r[8];
    kb_load32(seed, seeds, i);
    sha512_prefixed<8>(d, seed, nullptr, 0);
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = d[k];
    a[0] &= 0xfffffff8u;                     // digest[0] &= 0xf8
    a[7] = (a[7] & 0x7fffffffu) | 0x40000000u;  // digest[31] &= 0x7f; |= 0x40   (unreduced scalar, SURVEY §A3)
    const uint64_t lo = msg_off[i], hi = msg_off[i + 1];
    uint32_t d2[16];
    sha512_prefixed<8>(d2, d + 8, msg + lo, hi - lo);   // prefix = digest[32..64]
    sc_reduce512(r, d2);
    int8_t e[64];
    ge_p3 h;
    sc_recode16(e, r);
    ge_scalarmult_base<true>(h, e, base);
    kb_store_xyz(xyz, 2 * i, h);
    sc_recode16(e, a);
    ge_scalarmult_base<true>(h, e, base);
    kb_store_xyz(xyz, 2 * i + 1, h);
    kb_store32(a_out, i, a);
    kb_store32(r_out, i, r);
}
static __global__ void __launch_bounds__(KB_THREADS) k_sign_finish(size_t n, const uint8_t* ra, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* a_in, const uint8_t* r_in, uint8_t* sig, uint8_t* pk)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t rw[8], aw[8], d[16], h[8], a[8], r[8], s[8];
    kb_load32(rw, ra, 2 * i);
    kb_load32(aw, ra, 2 * i + 1);
    const uint64_t lo = msg_off[i], hi = msg_off[i + 1];
    sha512_ram(d, rw, aw, msg + lo, hi - lo);
    sc_reduce512(h, d);
    kb_load32(a, a_in, i);
    kb_load32(r, r_in, i);
    sc_muladd(s, h, a, r);
    kb_store32(sig, 2 * i, rw);
    kb_store32(sig, 2 * i + 1, s);
    if (pk) kb_store32(pk, i, aw);
}

#endif  // KB_K_SIGN
// ---- eddsa::verify_with_checks / schnorr::verify_with_checks, two launches (ops.cuh: sig_stage1 / sig_finish)
#ifndef KB_VERIFY_MINBLOCKS
#define KB_VERIFY_MINBLOCKS 3
#endif
template <bool SCHNORR>
static __global__ void __launch_bounds__(KB_THREADS, KB_VERIFY_MINBLOCKS) k_verify_stage1(size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, uint64_t msg_base, const uint8_t* sig, uint32_t* xyz, uint8_t* flags,
                                                              const ge_precomp* table128)
{
    __shared__ uint4 base_raw[128 * 24 / 4];
    ge_precomp* base128 = reinterpret_cast<ge_precomp*>(base_raw);
    kb_stage(reinterpret_cast<uint32_t*>(base128), reinterpret_cast<const uint32_t*>(table128), 128 * 24);
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n;   // tail threads redo the last item so that they reach the block barriers
    if (!live) i = n - 1;
    uint32_t pw[8], sw[16];
    ge_cached tbl[8];
    kb_load32(pw, pk, i);
    kb_load32(sw, sig, 2 * i);
    kb_load32(sw + 8, sig, 2 * i + 1);
    // msg_off holds offsets into the caller's whole message array; `msg` points at byte msg_base of it
    const uint64_t lo = msg_off[i], hi = msg_off[i + 1];
    ge_p3 Q;
    const uint32_t f = sig_stage1<SCHNORR>(Q, pw, sw, msg + (lo - msg_base), hi - lo, base128, tbl);
    if (live) {
        kb_store_xyz(xyz, i, Q);
        flags[i] = (uint8_t)f;
    }
}
template <bool SCHNORR>
static __global__ void __launch_bounds__(KB_THREADS) k_verify_stage2(size_t n, const uint32_t* xyz, const uint8_t* flags, const uint8_t* sig, uint8_t* status)
{
    kb_batch_compress(n, xyz, [&](size_t i, uint32_t* enc) {
        uint32_t rw[8];
        kb_load32(rw, sig, 2 * i);
        status[i] = (uint8_t)sig_finish<SCHNORR>(flags[i], enc, rw);
    });
}

#if defined(KB_K_KEYSET)
// ---- key sets (ops.cuh kb_key_*, sig_keyset_stage1): verification under registered public keys.  A key set holds, per key,
// its 32-byte encoding, one byte of facts (kb_key_facts) and its comb of KB_KEY_ENTRIES affine entries.
// One thread per (key, comb position).
static __global__ void __launch_bounds__(KB_THREADS) k_keyset_build(size_t nkeys, const uint8_t* pk, uint8_t* facts, ge_precomp* ktab)
{
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nkeys * KB_KEY_POS) return;
    const size_t k = t / KB_KEY_POS;
    const int p = (int)(t % KB_KEY_POS);
    uint32_t pw[8];
    kb_load32(pw, pk, k);
    ge_p3 A;
    const uint32_t f = kb_key_facts(A, pw);
    if (p == 0) facts[k] = (uint8_t)f;
    kb_key_row(ktab + k * KB_KEY_ENTRIES + (size_t)p * KB_KEY_HALF, A, p);
}
// sig_stage1 of signature i under key key_idx[i]: (X, Y, Z) and the flag byte in the layout of k_verify_stage1, for
// k_verify_stage2.  An index outside the key set reads nothing of it; the item is off the fast path and
// k_keyset_bad_index overwrites its status.
template <bool SCHNORR>
static __global__ void __launch_bounds__(KB_THREADS) k_keyset_verify(size_t n, const uint32_t* key_idx, size_t nkeys, const uint8_t* kpk, const uint8_t* facts, const ge_precomp* ktab,
                                                                     const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, const ge_precomp* comb, uint32_t* xyz, uint8_t* flags)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t k = __ldg(key_idx + i);
    uint32_t pw[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sw[16], kf = 0;
    const ge_precomp* kt = nullptr;
    if (k < nkeys) {
        kb_load32(pw, kpk, k);
        kf = __ldg(facts + k);
        kt = ktab + (size_t)k * KB_KEY_ENTRIES;
    }
    kb_load32(sw, sig, 2 * i);
    kb_load32(sw + 8, sig, 2 * i + 1);
    const uint64_t lo = msg_off[i], hi = msg_off[i + 1];
    ge_p3 Q;
    const uint32_t f = sig_keyset_stage1<SCHNORR>(Q, kf, pw, sw, msg + lo, hi - lo, comb, kt);
    kb_store_xyz(xyz, i, Q);
    flags[i] = (uint8_t)f;
}
// status 0xFF for every item whose key index is outside the key set (runs after k_verify_stage2)
static __global__ void __launch_bounds__(256) k_keyset_bad_index(size_t n, const uint32_t* key_idx, size_t nkeys, uint8_t* status)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && __ldg(key_idx + i) >= nkeys) status[i] = 0xFF;
}
// k_keyset_verify<true> for one signature batch of a DKG round (kb_dkg_process_round_keyed).  Item k = (d - dealer_lo) n + i
// is signed by dealer dealer_lo + k / n (a deal, RESP = false) or by verifier k % n (a response, RESP = true); the caller
// has checked that every such key is in the set, so no index array is read.  msg_off holds offsets into the caller's
// whole message array; `msg` points at byte msg_base of it.
template <bool RESP>
static __global__ void __launch_bounds__(KB_THREADS) k_keyset_verify_round(size_t m, size_t n, size_t dealer_lo, const uint8_t* kpk, const uint8_t* facts, const ge_precomp* ktab,
                                                                           const uint8_t* msg, const uint64_t* msg_off, uint64_t msg_base, const uint8_t* sig, const ge_precomp* comb,
                                                                           uint32_t* xyz, uint8_t* flags)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const size_t k = RESP ? i % n : dealer_lo + i / n;
    uint32_t pw[8], sw[16];
    kb_load32(pw, kpk, k);
    const uint32_t kf = __ldg(facts + k);
    kb_load32(sw, sig, 2 * i);
    kb_load32(sw + 8, sig, 2 * i + 1);
    const uint64_t lo = msg_off[i], hi = msg_off[i + 1];
    ge_p3 Q;
    const uint32_t f = sig_keyset_stage1<true>(Q, kf, pw, sw, msg + (lo - msg_base), hi - lo, comb, ktab + k * KB_KEY_ENTRIES);
    kb_store_xyz(xyz, i, Q);
    flags[i] = (uint8_t)f;
}
// ---- Point::mul(s, Some(A)) for registered keys: item i = scalars[i] * keys[key_idx[i]] (ops.cuh kb_keyset_mul_one), (X, Y, Z)
// in the layout of k_mul for k_compress_batch with status as its `bad` array.  An index outside the key set reads nothing of
// it and gives the identity with status 0xFF.  No block barrier: items of one block take different paths.
template <bool CT>
static __global__ void __launch_bounds__(KB_THREADS) k_keyset_mul(size_t n, const uint32_t* key_idx, size_t nkeys, const uint8_t* kpk, const uint8_t* facts, const ge_precomp* ktab,
                                                                  const uint8_t* scalars, uint32_t* xyz, uint8_t* status)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t k = __ldg(key_idx + i);
    ge_p3 h;
    uint32_t st = 0xFF;
    if (k < nkeys) {
        uint32_t s[8], pw[8];
        int8_t e[64];
        kb_load32(s, scalars, i);
        kb_load32(pw, kpk, k);
        sc_recode16(e, s);
        st = kb_keyset_mul_one<CT>(h, __ldg(facts + k), pw, e, ktab + (size_t)k * KB_KEY_ENTRIES);
    } else {
        ge_identity(h);
    }
    kb_store_xyz(xyz, i, h);
    status[i] = (uint8_t)st;
}
#endif  // KB_K_KEYSET

// ---- the same verifiers with half-size scalars (ops.cuh sig_half_*, half.cuh): 128 doublings per signature,
// verdict from a projective identity test (no inversion).  Two launches so that the two phases — which have
// very different code (decompression / SHA-512 / Euclid vs. the doubling loop) and register needs — do not
// compete for the instruction cache on one SM:
//   k_verify_half_prep   checks, decompress A and R, h, (u, v), u*s mod L   -> a record per signature
//   k_verify_half_main   digit strings, two tables, the 33-window loop        -> status
// The record of one signature, KB_HALF_REC_WORDS 32-bit words, written and read only through the accessors below.  It
// crosses HBM exactly once, so its accesses are streaming (__stcs / __ldcs; the sort reads u and v through __ldg):
//   words  0 .. 23   -A as affine X, Y, T             words 24 .. 47   -R as affine X, Y, T
//   words 48 .. 71   u*s mod L, u, |v|
//   word  72         flags | window count << 8 | sign(v) << 16 (the main kernel turns -A into A' = -sign(v) A)
//   word  73         the "decodes" bits of the split preparation (bit 0: A, bit 1: R)
#define KB_HALF_REC_WORDS 76
__device__ __forceinline__ uint32_t* kb_rec_at(uint32_t* recs, size_t i) { return recs + KB_HALF_REC_WORDS * i; }
__device__ __forceinline__ const uint32_t* kb_rec_at(const uint32_t* recs, size_t i) { return recs + KB_HALF_REC_WORDS * i; }
// point part k: -A (k = 0) or -R (k = 1)
__device__ __forceinline__ void kb_rec_store_point(uint32_t* o, int k, const fe& x, const fe& y, const fe& t)
{
    kb_store_fe_cs(o + 24 * k, x);
    kb_store_fe_cs(o + 24 * k + 8, y);
    kb_store_fe_cs(o + 24 * k + 16, t);
}
__device__ __forceinline__ void kb_rec_store_scalars(uint32_t* o, const kb_half_sc& sc)
{
    uint4* q = reinterpret_cast<uint4*>(o + 48);
    __stcs(q + 0, make_uint4(sc.w[0], sc.w[1], sc.w[2], sc.w[3]));
    __stcs(q + 1, make_uint4(sc.w[4], sc.w[5], sc.w[6], sc.w[7]));
    __stcs(q + 2, make_uint4(sc.u[0], sc.u[1], sc.u[2], sc.u[3]));
    __stcs(q + 3, make_uint4(sc.u[4], sc.u[5], sc.u[6], sc.u[7]));
    __stcs(q + 4, make_uint4(sc.v[0], sc.v[1], sc.v[2], sc.v[3]));
    __stcs(q + 5, make_uint4(sc.v[4], sc.v[5], sc.v[6], sc.v[7]));
}
__device__ __forceinline__ uint32_t kb_rec_pack72(uint32_t f, int nwin, uint32_t vneg) { return f | ((uint32_t)nwin << 8) | (vneg << 16); }
__device__ __forceinline__ uint32_t kb_rec_flags72(uint32_t w72) { return w72 & 0xffu; }
__device__ __forceinline__ uint32_t kb_rec_rest72(uint32_t w72) { return w72 & 0x1ff00u; }   // window count, sign(v) in place
__device__ __forceinline__ void kb_rec_unpack72(uint32_t w72, uint32_t& f, int& nwin, uint32_t& vneg)
{
    f = kb_rec_flags72(w72);
    nwin = (int)((w72 >> 8) & 0xffu);
    vneg = (w72 >> 16) & 1u;
}
// word 72 alone: the split preparation's scalars kernel, which leaves word 73 to the points kernel
__device__ __forceinline__ void kb_rec_store72(uint32_t* o, uint32_t w72) { __stcs(o + 72, w72); }
__device__ __forceinline__ void kb_rec_store73(uint32_t* o, uint32_t dec) { __stcs(o + 73, dec); }
// the last store of a preparation: word 72 in one 16-byte store that clears words 73 .. 75
__device__ __forceinline__ void kb_rec_store72_clear73(uint32_t* o, uint32_t w72) { __stcs(reinterpret_cast<uint4*>(o + 72), make_uint4(w72, 0u, 0u, 0u)); }
__device__ __forceinline__ void kb_rec_load72_73(const uint32_t* o, uint32_t& w72, uint32_t& dec)
{
    const uint4 a = __ldcs(reinterpret_cast<const uint4*>(o + 72));
    w72 = a.x;
    dec = a.y;
}
// what a signature off the fast path hands to the main kernel: operands (0, 1, 0) and scalars 0 (word 72 is the caller's)
__device__ __forceinline__ void kb_rec_store_neutral(uint32_t* o)
{
    const uint4 z = make_uint4(0u, 0u, 0u, 0u), one = make_uint4(1u, 0u, 0u, 0u);
    uint4* r = reinterpret_cast<uint4*>(o);
    KB_UNROLL
    for (int k = 0; k < 12; k++) __stcs(r + k, (k == 2 || k == 8) ? one : z);
    uint4* q = reinterpret_cast<uint4*>(o + 48);
    KB_UNROLL
    for (int k = 0; k < 6; k++) __stcs(q + k, z);
}
// u and v, for the sort by loop length
__device__ __forceinline__ void kb_rec_load_uv(uint32_t* u, uint32_t* v, const uint32_t* o)
{
    const uint4* q = reinterpret_cast<const uint4*>(o + 48);
    uint4 a;
    a = __ldg(q + 2); u[0] = a.x; u[1] = a.y; u[2] = a.z; u[3] = a.w;
    a = __ldg(q + 3); u[4] = a.x; u[5] = a.y; u[6] = a.z; u[7] = a.w;
    a = __ldg(q + 4); v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    a = __ldg(q + 5); v[4] = a.x; v[5] = a.y; v[6] = a.z; v[7] = a.w;
}
// the whole record, with A' = -sign(v) A in place of -A
__device__ __forceinline__ void kb_rec_load(kb_half_rec& rec, const uint32_t* o)
{
    kb_load_fe_cs(rec.ax, o);
    kb_load_fe_cs(rec.ay, o + 8);
    kb_load_fe_cs(rec.at, o + 16);
    kb_load_fe_cs(rec.rx, o + 24);
    kb_load_fe_cs(rec.ry, o + 32);
    kb_load_fe_cs(rec.rt, o + 40);
    const uint4* q = reinterpret_cast<const uint4*>(o + 48);
    uint4 a;
    a = __ldcs(q + 0); rec.w[0] = a.x; rec.w[1] = a.y; rec.w[2] = a.z; rec.w[3] = a.w;
    a = __ldcs(q + 1); rec.w[4] = a.x; rec.w[5] = a.y; rec.w[6] = a.z; rec.w[7] = a.w;
    a = __ldcs(q + 2); rec.u[0] = a.x; rec.u[1] = a.y; rec.u[2] = a.z; rec.u[3] = a.w;
    a = __ldcs(q + 3); rec.u[4] = a.x; rec.u[5] = a.y; rec.u[6] = a.z; rec.u[7] = a.w;
    a = __ldcs(q + 4); rec.v[0] = a.x; rec.v[1] = a.y; rec.v[2] = a.z; rec.v[3] = a.w;
    a = __ldcs(q + 5); rec.v[4] = a.x; rec.v[5] = a.y; rec.v[6] = a.z; rec.v[7] = a.w;
    a = __ldcs(q + 6);
    uint32_t vneg;
    kb_rec_unpack72(a.x, rec.f, rec.nwin, vneg);
    sig_half_apply_vneg(rec.ax, rec.at, vneg);
}
#ifndef KB_VERIFY_PREP_MINBLOCKS
#define KB_VERIFY_PREP_MINBLOCKS 5
#endif
// The two phases of the preparation load different pipes: the decompressions are multiplier-bound (IMAD.WIDE), the
// hash and the lattice step ALU-bound, and blocks that start together on an SM stay in step for the whole launch.
// -DKB_PREP_ROLES=1 lets every block draw its phase order from a counter of the SM it runs on (half of an SM's blocks
// decompress while the other half hash).  MEASURED (round 2, 2^20 signatures): 5.96 ms against 4.97 ms with one phase
// order — warps on different code paths miss the instruction cache more than the idle pipe costs; kept as a build
// option only.  Each phase writes its part of the record straight to memory; only the flags, sign(v) and the window
// count stay in registers across phases (312 -> 180 bytes of spill stores).
#ifndef KB_PREP_ROLES
#define KB_PREP_ROLES 0
#endif
#ifndef KB_PREP_SYNC
#define KB_PREP_SYNC 1
#endif
#if KB_PREP_ROLES
static __device__ unsigned int kb_prep_role_counter[1024];
#endif
template <bool SCHNORR>
static __global__ void __launch_bounds__(KB_THREADS, KB_VERIFY_PREP_MINBLOCKS) k_verify_half_prep(size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, uint64_t msg_base, const uint8_t* sig, uint32_t* recs)
{
    int role = 0;
#if KB_PREP_ROLES
    __shared__ unsigned int s_role;
    if (threadIdx.x == 0) {
        unsigned int smid;
        asm("mov.u32 %0, %%smid;" : "=r"(smid));
        s_role = atomicAdd(&kb_prep_role_counter[smid & 1023u], 1u);
    }
    __syncthreads();
    role = (int)(s_role & 1u);
#endif
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
#if KB_PREP_SYNC
    if (i >= n) i = n - 1;   // tail threads redo the last item (same values, same address) so that they reach the barriers
#else
    if (i >= n) return;
#endif
    uint32_t pw[8], sw[16];
    kb_load32(pw, pk, i);
    kb_load32(sw, sig, 2 * i);
    kb_load32(sw + 8, sig, 2 * i + 1);
    uint32_t* o = kb_rec_at(recs, i);
    uint32_t dec = 0, f = 0, vneg = 0;
    int nwin = 0;
    KB_NOUNROLL
    for (int pass = 0; pass < 2; pass++) {
#if KB_PREP_SYNC
        __syncthreads();
#endif
        if ((pass ^ role) == 0) {
            // one copy of the decompression code for both points
            KB_NOUNROLL
            for (int k = 0; k < 2; k++) {
#if KB_PREP_SYNC
                __syncthreads();
#endif
                fe x, y, t;
                dec |= sig_half_point(x, y, t, k ? sw : pw) << k;
                kb_rec_store_point(o, k, x, y, t);
            }
        } else {
            // msg_off holds offsets into the caller's whole message array; `msg` points at byte msg_base of it
            const uint64_t lo = msg_off[i], hi = msg_off[i + 1];
            kb_half_sc sc;
            sig_half_scalars<SCHNORR>(sc, pw, sw, msg + (lo - msg_base), hi - lo);
            kb_rec_store_scalars(o, sc);
            f = sc.f;
            vneg = sc.vneg;
            nwin = sc.nwin;
        }
    }
    f = sig_half_flags<SCHNORR>(f, dec);
    if (!(f & KB_F_FAST)) {
        kb_rec_store_neutral(o);   // off the fast path (rare): neutral operands, no windows
        nwin = 0;
        vneg = 0;
    }
    kb_rec_store72_clear73(o, kb_rec_pack72(f, nwin, vneg));
}
// ---- the preparation as TWO kernels that share the SMs (KB_VERIFY_SPLIT=1, capi_verify.cu).  The phases of
// k_verify_half_prep load different pipes and run one after the other in every block; here the "scalars" phase is a
// PERSISTENT kernel of a few blocks per SM (work drawn from a counter) that is launched first on a side stream, and the
// "points" phase an ordinary grid that fills what is left of every SM: warps of both kinds are resident at all times, the
// ALU-bound ones issue into the slots the multiplier-bound ones leave empty.  The verdict bits of both meet in
// k_verify_half_fix (word 72 / 73 of the record), which also neutralises the records that are off the fast path — the
// main kernel reads the same record layout from either preparation.
template <int MINB>
static __global__ void __launch_bounds__(KB_THREADS, MINB) k_verify_half_points(size_t n, const uint8_t* pk, const uint8_t* sig, uint32_t* recs)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) i = n - 1;   // tail threads redo the last item (same values, same address) so that they reach the barriers
    uint32_t* o = kb_rec_at(recs, i);
    uint32_t dec = 0;
    KB_NOUNROLL
    for (int k = 0; k < 2; k++) {
        __syncthreads();
        uint32_t w[8];
        if (k) kb_load32(w, sig, 2 * i);
        else kb_load32(w, pk, i);
        fe x, y, t;
        dec |= sig_half_point(x, y, t, w) << k;
        kb_rec_store_point(o, k, x, y, t);
    }
    kb_rec_store73(o, dec);
}
template <bool SCHNORR>
static __global__ void __launch_bounds__(KB_THREADS, 4) k_verify_half_scalars(size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, uint64_t msg_base, const uint8_t* sig, uint32_t* recs,
                                                                              unsigned long long* counter)
{
    __shared__ unsigned long long s_base;
    for (;;) {
        if (threadIdx.x == 0) s_base = atomicAdd(counter, (unsigned long long)blockDim.x);
        __syncthreads();
        const size_t base = (size_t)s_base;
        __syncthreads();
        if (base >= n) return;
        const size_t i = base + threadIdx.x;
        if (i >= n) continue;
        uint32_t pw[8], sw[16];
        kb_load32(pw, pk, i);
        kb_load32(sw, sig, 2 * i);
        kb_load32(sw + 8, sig, 2 * i + 1);
        const uint64_t lo = msg_off[i], hi = msg_off[i + 1];
        kb_half_sc sc;
        sig_half_scalars<SCHNORR>(sc, pw, sw, msg + (lo - msg_base), hi - lo);
        uint32_t* o = kb_rec_at(recs, i);
        kb_rec_store_scalars(o, sc);
        kb_rec_store72(o, kb_rec_pack72(sc.f, sc.nwin, sc.vneg));
    }
}
template <bool SCHNORR>
static __global__ void __launch_bounds__(256) k_verify_half_fix(size_t n, uint32_t* recs)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t* o = kb_rec_at(recs, i);
    uint32_t w72, dec;
    kb_rec_load72_73(o, w72, dec);
    const uint32_t f = sig_half_flags<SCHNORR>(kb_rec_flags72(w72), dec);
    uint32_t rest = kb_rec_rest72(w72);
    if (!(f & KB_F_FAST)) {
        kb_rec_store_neutral(o);   // off the fast path (rare): neutral operands, no windows
        rest = 0;
    }
    kb_rec_store72_clear73(o, f | rest);
}
// ---- order of the records for the main kernel: a counting sort by the number of digit pairs each needs (the same
// sc_joint4_pairs the main kernel takes its trip count from), longest first.  2^20 honest signatures need 60 .. 68
// pairs, 64.6 on average; a block of 128 random ones runs the maximum of its members, 66.4 on average.
#define KB_SORT_BINS 129
#if KB_HALF_JOINT
static __global__ void __launch_bounds__(256) k_half_sort_count(size_t n, const uint32_t* recs, uint8_t* keys, uint32_t* hist)
{
    __shared__ uint32_t s_hist[KB_SORT_BINS];
    for (int k = threadIdx.x; k < KB_SORT_BINS; k += blockDim.x) s_hist[k] = 0;
    __syncthreads();
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        uint32_t u[8], v[8];
        kb_rec_load_uv(u, v, kb_rec_at(recs, i));
        const int key = sc_joint4_pairs(u, v);   // 1 .. 128
        keys[i] = (uint8_t)key;
        atomicAdd(&s_hist[key], 1u);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < KB_SORT_BINS; k += blockDim.x)
        if (s_hist[k]) atomicAdd(&hist[k], s_hist[k]);
}
// first position of every bin, longest records first
static __global__ void k_half_sort_scan(const uint32_t* hist, uint32_t* cursor)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t pos = 0;
    for (int k = KB_SORT_BINS - 1; k >= 0; k--) {
        cursor[k] = pos;
        pos += hist[k];
    }
}
static __global__ void __launch_bounds__(256) k_half_sort_scatter(size_t n, const uint8_t* keys, uint32_t* cursor, uint32_t* perm)
{
    __shared__ uint32_t s_cnt[KB_SORT_BINS], s_base[KB_SORT_BINS];
    for (int k = threadIdx.x; k < KB_SORT_BINS; k += blockDim.x) s_cnt[k] = 0;
    __syncthreads();
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t key = 0, rank = 0;
    if (i < n) {
        key = keys[i];
        rank = atomicAdd(&s_cnt[key], 1u);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < KB_SORT_BINS; k += blockDim.x)
        if (s_cnt[k]) s_base[k] = atomicAdd(&cursor[k], s_cnt[k]);
    __syncthreads();
    if (i < n) perm[s_base[key] + rank] = (uint32_t)i;
}
#endif
// Resident blocks per SM of the main kernel.  3 (168 registers, no spills) was the best setting while two radix-16 tables
// sat in local memory (2 blocks: +5 %, 4: slower in round 1); with the joint table (1.7 KB per thread, a third of the DRAM
// traffic) 4 blocks (128 registers, 208 bytes of spills) win: 14.82 -> 14.51 ms for 2^20 signatures (profiles/r2_ab_sync1_mb4.txt).
#ifndef KB_VERIFY_HALF_MINBLOCKS
#define KB_VERIFY_HALF_MINBLOCKS 4
#endif
#ifndef KB_HALF_PREFETCH
#define KB_HALF_PREFETCH 1   // operands of the additions fetched one step ahead (ops.cuh ge_triple_scalarmult_prefetch)
#endif
template <bool SCHNORR>
static __global__ void __launch_bounds__(KB_THREADS, KB_VERIFY_HALF_MINBLOCKS) k_verify_half_main(size_t n, const uint32_t* recs, const uint32_t* perm, uint8_t* status, const ge_precomp* comb, int min_windows)
{
    __shared__ int s_nwin;
#if KB_HALF_JOINT
    if (threadIdx.x == 0) s_nwin = 2 * min_windows;   // the joint loop counts radix-4 digit pairs
#else
    if (threadIdx.x == 0) s_nwin = min_windows;   // KB_HALF_MIN_WINDOWS, or more when a test forces long loops
#endif
    __syncthreads();
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n;   // tail threads redo the last item so that they reach the block barriers
    if (!live) i = n - 1;
    if (perm) i = perm[i];     // the order of k_half_sort_*: records of like loop length share a block
    kb_half_rec rec;
    kb_rec_load(rec, kb_rec_at(recs, i));
    kb_comb_digit dw[KB_COMB_POS];
#if KB_HALF_JOINT
    ge_cached tbl[KB_JOINT_SLOTS];
    uint32_t uk[8], vk[8];
    sig_half_setup_joint(dw, uk, vk, tbl, rec);
#else
    ge_cached tbl[16];
    int8_t eu[64], ev[64];
    sig_half_setup(dw, eu, ev, tbl, rec);
#endif
    // the window count of the block = the longest any of its signatures needs
#if KB_HALF_JOINT
    int nwin = __reduce_max_sync(0xffffffffu, sc_joint4_pairs(rec.u, rec.v));
#else
    int nwin = __reduce_max_sync(0xffffffffu, rec.nwin);
#endif
    if ((threadIdx.x & 31) == 0) atomicMax(&s_nwin, nwin);
    __syncthreads();
    nwin = s_nwin;
    ge_p3 W;
#if KB_HALF_JOINT
    ge_triple_scalarmult_joint(W, nwin, dw, uk, vk, tbl, comb);
#elif KB_HALF_PREFETCH
    ge_triple_scalarmult_prefetch(W, nwin, dw, eu, ev, tbl, comb);
#else
    ge_triple_scalarmult_vartime(W, nwin, dw, eu, ev, tbl, comb);
#endif
    if (live) status[i] = (uint8_t)sig_half_finish<SCHNORR>(rec.f, W);
}

#if defined(KB_K_POLY)
// ---- committed polynomials
// commitments -> cached operand form, 32 words per commitment; bad[c] = 1 if undecodable
static __global__ void __launch_bounds__(KB_THREADS) k_commit_prepare(size_t ncommit, const uint8_t* commits, uint32_t* cached, uint8_t* bad)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ncommit) return;
    uint32_t w[8];
    kb_load32(w, commits, i);
    ge_p3 p;
    const uint32_t ok = ge_decompress(p, w);
    ge_cached c;
    ge_to_cached(c, p);
    kb_store_cached_w128(cached + 32 * i, c);
    bad[i] = (uint8_t)(ok ^ 1u);
}
// the same from the reference's in-memory / serde form (40 limbs per point, ge.cuh kb_point_from_limbs_checked)
static __global__ void __launch_bounds__(KB_THREADS) k_commit_prepare_limbs(size_t ncommit, const int32_t* limbs, uint32_t* cached, uint8_t* bad)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ncommit) return;
    ge_p3 p;
    const uint32_t ok = kb_point_from_limbs_checked(p, limbs + 40 * i);
    if (!ok) ge_identity(p);
    ge_cached c;
    ge_to_cached(c, p);
    kb_store_cached_w128(cached + 32 * i, c);
    bad[i] = (uint8_t)(ok ^ 1u);
}
// PriPoly::eval (share/poly.rs:133-141) for every (polynomial d, index i): out[d * n + i] = sum_j coeffs[d][j] (i+1)^j mod L
// by Horner's rule with sc_mul_add — the dealer's side of a round (new_dealer, share/vss/pedersen/vss.rs:313: f.eval(i) for
// all i).  The coefficients are secret: sc_muladd is branch-free and the evaluation point is public.
static __global__ void __launch_bounds__(KB_THREADS) k_pripoly_eval(size_t npoly, size_t t, const uint8_t* coeffs, size_t n, uint8_t* out)
{
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= npoly * n) return;
    const size_t d = k / n, i = k % n;
    uint32_t x[8] = {0, 0, 0, 0, 0, 0, 0, 0}, v[8] = {0, 0, 0, 0, 0, 0, 0, 0}, c[8];
    const uint64_t xv = (uint64_t)i + 1;
    x[0] = (uint32_t)xv;
    x[1] = (uint32_t)(xv >> 32);
    for (size_t j = t; j-- > 0;) {
        kb_load32(c, coeffs, d * t + j);
        sc_muladd(v, v, x, c);
    }
    kb_store32(out, k, v);
}
// PubPoly::eval (poly.rs:457-469) and, with shares != nullptr, the verify_deal comparison
// (vss/pedersen/vss.rs:899-912).  Item k is (poly_id[k], idx[k]); with poly_id == nullptr the
// items enumerate a DKG round: k = i * npoly + d (verifier-major), so the 32 lanes of a warp
// hold 32 different dealers and the SAME evaluation point x = i + 1 — the double-and-add over
// the bits of x is then branch-uniform across the warp.
static __global__ void __launch_bounds__(KB_THREADS) k_poly_eval(size_t m, size_t npoly, size_t t, const uint32_t* cached, const uint8_t* bad, const uint32_t* poly_id,
                                                          const uint32_t* idx, size_t n_verifiers, const uint8_t* shares, uint32_t* xyz, uint8_t* status, uint8_t* verdict, const ge_precomp* table)
{
    extern __shared__ uint4 smem4[];
    ge_precomp* base = reinterpret_cast<ge_precomp*>(smem4);
    if (shares) kb_stage(reinterpret_cast<uint32_t*>(base), reinterpret_cast<const uint32_t*>(table), 64 * 8 * 24);
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = k < m;   // the coefficient loop holds a block barrier: tail threads redo the last item
    if (!live) k = m - 1;
    size_t d, i, slot;
    if (poly_id) {
        d = poly_id[k];
        i = idx[k];
        slot = k;
    } else {
        d = k % npoly;
        i = k / npoly;
        slot = d * n_verifiers + i;
    }
    const uint32_t* cp = cached + 32 * (d * t);
    const uint8_t* bp = bad + d * t;
    ge_p3 v;
    ge_identity(v);
    uint32_t anybad = 0;
    kb_naf xn;
    kb_naf_from(xn, (uint64_t)i + 1);
    for (size_t j = t; j-- > 0;) {
        __syncthreads();   // keeps the block's warps on the same instructions (see KB_LOCKSTEP in ops.cuh)
        ge_cached c;
        kb_load_cached_w128(c, cp + 32 * j);
        anybad |= bp[j];
        kb_horner_step(v, xn, c);
    }
    if (!shares) {
        if (!live) return;
        if (anybad) ge_identity(v);
        kb_store_xyz(xyz, slot, v);
        status[slot] = (uint8_t)anybad;
        return;
    }
    uint32_t s[8];
    int8_t e[64];
    kb_load32(s, shares, slot);
    sc_recode16(e, s);
    ge_p3 h;
    ge_scalarmult_base<true>(h, e, base);
    // Point::eq compares canonical encodings (point.rs:227): equal affine points <=> X1 Z2 = X2 Z1 and
    // Y1 Z2 = Y2 Z1 (Z never vanishes on the curve), so no inversion is needed for a verdict.
    fe l, r, df;
    fe_mul(l, v.X, h.Z);
    fe_mul(r, h.X, v.Z);
    fe_sub(df, l, r);
    uint32_t same = fe_is_zero(df);
    fe_mul(l, v.Y, h.Z);
    fe_mul(r, h.Y, v.Z);
    fe_sub(df, l, r);
    same &= fe_is_zero(df);
    if (live) verdict[slot] = (uint8_t)(same & (anybad ^ 1u));
}

#endif  // KB_K_POLY
// ---- integer-multiply roofline probe
template <int KIND>
static __global__ void __launch_bounds__(256) k_probe(int iters, uint32_t seed, uint32_t* sink)
{
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (KIND == 0) {
        // 8 independent 64-bit accumulators: acc += lo32(acc) * b — one IMAD.WIDE.U32 per step and nothing else
        // (the multiplicand is the accumulator's own low word, so the compiler can neither hoist the product nor
        // has to spend an ALU instruction on making it vary)
        uint64_t acc[8];
        uint32_t b = (seed * 2654435761u + tid) | 1u;
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = ((uint64_t)(seed ^ tid) << 32) | (tid + 977u * k + 1u);
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int k = 0; k < 8; k++) acc[k] = (uint64_t)(uint32_t)acc[k] * b + acc[k];
        }
        uint64_t x = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) x ^= acc[k];
        if (x == 0x1234567u) sink[0] = (uint32_t)x;
    } else if (KIND == 1) {
        // 8 independent 32-bit accumulators: acc = acc * b + a  (IMAD)
        uint32_t acc[8];
        uint32_t a = seed ^ tid, b = (seed * 2654435761u + tid) | 1u;
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = tid + k;
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int k = 0; k < 8; k++) acc[k] = acc[k] * b + a;
        }
        uint32_t x = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) x ^= acc[k];
        if (x == 0x1234567u) sink[0] = x;
    } else if (KIND == 2) {
        // two independent 4-product carry chains per iteration (the fe_mul inner pattern)
        uint32_t e[9], o[9];
#pragma unroll
        for (int k = 0; k < 9; k++) { e[k] = tid + k; o[k] = seed + k; }
        uint32_t a0 = seed ^ tid, a1 = a0 * 3u, a2 = a0 * 5u, a3 = a0 * 7u, b = seed + 0x9e3779b9u;
        for (int it = 0; it < iters; it++) {
            kb_cmad4(e, a0, a1, a2, a3, b, e[8]);
            kb_cmad4(o, a1, a2, a3, a0, b, o[8]);
            b += e[0];
        }
        uint32_t x = 0;
#pragma unroll
        for (int k = 0; k < 9; k++) x ^= e[k] ^ o[k];
        if (x == 0x1234567u) sink[0] = x;
    } else {
        // the library's own field multiplication, two independent chains
        fe x, y, z;
#pragma unroll
        for (int k = 0; k < 8; k++) { x.v[k] = tid * 977u + k; y.v[k] = seed + 31u * k; z.v[k] = tid + seed * k; }
        for (int it = 0; it < iters; it++) {
            fe_mul(x, x, y);
            fe_mul(z, z, y);
        }
        uint32_t acc = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) acc ^= x.v[k] ^ z.v[k];
        if (acc == 0x1234567u) sink[0] = acc;
    }
}
