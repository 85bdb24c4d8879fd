// msm.cuh — Pippenger multi-scalar multiplication: out = sum_i s_i * P_i, the fold of
// Point::mul + Point::add (group/edwards25519/point.rs:179,207) that sits behind
// PubPoly::commit / recover_commit and the share verifiers.
//
// Pipeline (all on device, per chunk of <= 2^22 points):
//   prepare : decompress P_i (ge.rs:124) to affine (y+x, y-x, 2dxy); effective scalar
//             (the reference's out-of-domain top-digit rule, SURVEY §A3) -> sign + magnitude
//   hist    : signed c-bit digits; per-bucket counts (atomicAdd)
//   scan    : exclusive prefix sum -> bucket offsets
//   scatter : counting sort of (point index, sign) into bucket order
//   accum   : LOAD-BALANCED bucket accumulation — every thread owns K consecutive sorted
//             entries (not one bucket), so skewed scalar distributions cannot starve the
//             grid; runs cut by a chunk boundary go to head/tail partials
//   merge   : stitch head/tail partials into their bucket
//   reduce  : per window, sum_k k * bucket_k by running sums over bucket groups
//   finish  : warp-shuffle tree over the group partials, then Horner over the windows
//
// Every stage body is a KB_FN taking an explicit thread id so tests/emu can run it on the
// host; only the warp-shuffle tree in finish is GPU-only.
#pragma once
#include "ge.cuh"
#include "poly.cuh"
#include "sc.cuh"

#define KB_MSM_CHUNK (1u << 22)
#define KB_MSM_GROUPS 4096  // most bucket groups per window in the reduction (scratch sizing; the driver picks 1024 or 2048)

#if defined(KB_HOST_EMU)
KB_FN uint32_t kb_atomic_add(uint32_t* p, uint32_t v) { uint32_t o = *p; *p = o + v; return o; }
#else
KB_FN uint32_t kb_atomic_add(uint32_t* p, uint32_t v) { return atomicAdd(p, v); }
#endif


struct kb_msm_plan {
    uint32_t n;        // points in this chunk
    uint32_t c;        // window bits
    uint32_t windows;  // ceil(257 / c)
    uint32_t half;     // 2^(c-1) buckets per window
    uint32_t nb;       // windows * half
    uint32_t k;        // sorted entries per accumulation thread (16..128, ~ the mean bucket size)
};

// entries per accumulation thread: about one mean bucket, so that most buckets are cut by at most one
// chunk boundary and the head/tail stitching stays cheap
static inline uint32_t kb_msm_chunk_entries(size_t n, uint32_t half)
{
    const size_t avg = n / half;
    uint32_t k = 16;
    while (k < 128 && k < avg) k <<= 1;
    return k;
}

static inline uint32_t kb_msm_window_bits_host(size_t n)
{
    uint32_t lg = 0;
    while ((n >> (lg + 1)) != 0) lg++;
    int c = (int)lg - 3;
    if (c < 4) c = 4;
    if (c > 16) c = 16;
    return (uint32_t)c;
}

// bucket groups per window in the reduction: fewer groups = longer serial runs in k_msm_reduce but a shorter fold in
// k_msm_window_sums (one block per window).  Measured (round 2, KB_MSM_GROUPS): 2^17 points 1.40 / 1.32 / 1.27 / 1.29 ms
// for 4096 / 2048 / 1024 / 512 groups, 2^22 points 14.76 / 14.66 / 14.68 / 14.86 ms.
// setting: the context's KB_MSM_GROUPS (0 = by window size); never more groups than buckets in a window.
static inline uint32_t kb_msm_groups_host(uint32_t half, uint32_t setting)
{
    const uint32_t gmax = setting ? setting : (half <= 8192u ? 1024u : 2048u);
    return half < gmax ? half : gmax;
}

// bits [pos, pos + c) of the 256-bit magnitude (zero beyond bit 255), c <= 16
KB_FN uint32_t sc_bits(const uint32_t* mag, uint32_t pos, uint32_t c)
{
    if (pos >= 256) return 0;
    const uint32_t wi = pos >> 5, sh = pos & 31;
    uint64_t v = mag[wi];
    if (wi + 1 < 8) v |= (uint64_t)mag[wi + 1] << 32;
    return (uint32_t)(v >> sh) & ((1u << c) - 1u);
}

// ---- prepare: point -> affine precomp (24 words); scalar -> magnitude (8 words) + sign
KB_FN void kb_msm_prepare_body(size_t i, const uint32_t* pw, const uint32_t* sw, uint32_t* pts, uint32_t* mags, uint8_t* negs, uint32_t* bad)
{
    ge_p3 p;
    const uint32_t ok = ge_decompress(p, pw);
    ge_precomp q;
    const fe d2 = KB_FE_D2;
    fe_add(q.ypx, p.Y, p.X);
    fe_sub(q.ymx, p.Y, p.X);
    fe_mul(q.xy2d, p.T, d2);
    if (!ok) {
        ge_precomp_identity(q);
        kb_atomic_add(bad, 1u);
    }
    kb_store_precomp_w32(pts + 24 * i, q);
    uint32_t mag[8], neg;
    sc_effective(mag, neg, sw);
    KB_UNROLL
    for (int k = 0; k < 8; k++) mags[8 * i + k] = mag[k];
    negs[i] = (uint8_t)neg;
}

// signed digits of one magnitude; calls f(w, bucket, sign) for every non-zero digit
template <typename F>
KB_FN void kb_msm_digits(const kb_msm_plan& pl, const uint32_t* mag, F f)
{
    uint32_t carry = 0;
    for (uint32_t w = 0; w < pl.windows; w++) {
        uint32_t d = sc_bits(mag, w * pl.c, pl.c) + carry;
        carry = 0;
        uint32_t sign = 0;
        if (d > pl.half) {
            d = (1u << pl.c) - d;
            sign = 1;
            carry = 1;
        }
        if (d != 0) f(w, w * pl.half + (d - 1), sign);
    }
}
KB_FN void kb_msm_hist_body(const kb_msm_plan& pl, size_t i, const uint32_t* mags, uint32_t* counts)
{
    kb_msm_digits(pl, mags + 8 * i, [&](uint32_t, uint32_t bucket, uint32_t) { kb_atomic_add(counts + bucket, 1u); });
}
KB_FN void kb_msm_scatter_body(const kb_msm_plan& pl, size_t i, const uint32_t* mags, const uint8_t* negs, const uint32_t* offsets, uint32_t* cursor, uint32_t* sorted)
{
    const uint32_t sneg = negs[i];
    kb_msm_digits(pl, mags + 8 * i, [&](uint32_t, uint32_t bucket, uint32_t sign) {
        const uint32_t slot = offsets[bucket] + kb_atomic_add(cursor + bucket, 1u);
        sorted[slot] = ((uint32_t)i << 1) | (sign ^ sneg);
    });
}

// ---- accum: thread t owns sorted entries [t*K, (t+1)*K)
// flags[t]: bit0 = head partial valid, bit1 = tail partial valid
// tailb[t]: the bucket of the tail partial (what k_msm_merge would otherwise have to search for)
KB_FN void kb_msm_accum_body(const kb_msm_plan& pl, size_t t, const uint32_t* offsets, const uint32_t* sorted, const uint32_t* pts, uint32_t* bucket_sum, uint32_t* heads,
                             uint32_t* tails, uint8_t* flags, uint32_t* tailb)
{
    const uint32_t total = offsets[pl.nb];
    const uint64_t s64 = (uint64_t)t * pl.k;
    flags[t] = 0;
    if (s64 >= total) return;
    const uint32_t s = (uint32_t)s64;
    const uint32_t e = (total - s < pl.k) ? total : s + pl.k;
    // bucket containing entry s: largest b with offsets[b] <= s (skipping empty buckets)
    uint32_t lo = 0, hi = pl.nb;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (offsets[mid] <= s) lo = mid;
        else hi = mid;
    }
    uint32_t b = lo;
    while (offsets[b + 1] <= s) b++;
    ge_p3 acc;
    ge_identity(acc);
    uint32_t fl = 0;
    uint32_t v = sorted[s];
    ge_precomp q;
    kb_load_precomp_w32(q, pts + 24 * (size_t)(v >> 1));
    for (uint32_t k = s; k < e; k++) {
        // fetch the NEXT entry's point before the ~900-instruction addition so the gather overlaps it.  (An additional
        // prefetch.global.L2 of the entry four ahead was measured SLOWER: 15.2 against 14.8 ms at 2^22.)
        const uint32_t vcur = v;
        ge_precomp qn;
        uint32_t vn = v;
        if (k + 1 < e) {
            vn = sorted[k + 1];
            kb_load_precomp_w32(qn, pts + 24 * (size_t)(vn >> 1));
        } else {
            qn = q;
        }
        ge_precomp_cneg(q, vcur & 1u);
        ge_madd<true>(acc, acc, q);
        q = qn;
        v = vn;
        const uint32_t bend = offsets[b + 1];
        if (k + 1 == bend || k + 1 == e) {
            // run of bucket b inside this chunk ends here
            const bool starts_before = offsets[b] < s;
            const bool ends_after = bend > e;
            if (starts_before) {
                kb_store_p3_w32(heads + 32 * t, acc);
                fl |= 1u;
            } else if (ends_after) {
                kb_store_p3_w32(tails + 32 * t, acc);
                tailb[t] = b;
                fl |= 2u;
            } else {
                kb_store_p3_w32(bucket_sum + 32 * (size_t)b, acc);
            }
            ge_identity(acc);
            if (k + 1 < e) {
                b++;
                while (offsets[b + 1] <= k + 1) b++;
            }
        }
    }
    flags[t] = (uint8_t)fl;
}

// ---- merge: thread t whose tail partial is valid owns that bucket: tail[t] + head[t+1] + ...
// Runs that continue over more than max_serial following chunks (skewed scalars; the top window
// of any reduced scalar set) are queued in long_list and summed by a whole warp (k_msm_merge_long).
// mode 0: both in one pass; 1: only queue the long runs; 2: only the short ones (the queue was filled by a mode-1 pass,
// so that the long and the short runs can be summed by two kernels side by side)
KB_FN void kb_msm_merge_body(const kb_msm_plan& pl, size_t t, size_t nthreads, const uint32_t* offsets, uint32_t max_serial, uint32_t* long_count, uint32_t* long_list,
                             uint32_t* bucket_sum, const uint32_t* heads, const uint32_t* tails, const uint8_t* flags, const uint32_t* tailb, int mode = 0)
{
    if (!(flags[t] & 2u)) return;
    const uint32_t b = tailb[t];   // the bucket of the last entry of chunk t (recorded by the accumulation)
    const uint32_t bend = offsets[b + 1];
    const size_t u_end = ((size_t)bend + pl.k - 1) / pl.k;  // chunks t+1 .. u_end-1 start inside the bucket
    if (u_end - (t + 1) > max_serial) {
        if (mode == 2) return;
        const uint32_t slot = kb_atomic_add(long_count, 1u);
        long_list[3 * slot] = (uint32_t)t;
        long_list[3 * slot + 1] = (uint32_t)u_end;
        long_list[3 * slot + 2] = b;
        return;
    }
    if (mode == 1) return;
    ge_p3 acc, h;
    kb_load_p3_w32(acc, tails + 32 * t);
    for (size_t u = t + 1; u < u_end && u < nthreads; u++) {
        if (flags[u] & 1u) {
            kb_load_p3_w32(h, heads + 32 * u);
            ge_cached hc;
            ge_to_cached(hc, h);
            ge_add<true>(acc, acc, hc);
        }
    }
    kb_store_p3_w32(bucket_sum + 32 * (size_t)b, acc);
}

// ---- reduce: group g of window w covers buckets [g*gs, (g+1)*gs) (0-based, bucket k has weight k+1)
//   run[w*G + g] = sum_k bucket_k                 over the group
//   tot[w*G + g] = sum_k (k - g*gs + 1) bucket_k   (running sum of running sums)
// so that the window sum is  sum_g tot_g + gs * sum_g g * run_g  (k_msm_window_sums).
KB_FN void kb_msm_reduce_body(const kb_msm_plan& pl, size_t tid, uint32_t groups, const uint32_t* offsets, const uint32_t* bucket_sum, uint32_t* part_run, uint32_t* part_tot)
{
    const uint32_t w = (uint32_t)(tid / groups), g = (uint32_t)(tid % groups);
    if (w >= pl.windows) return;
    const uint32_t gs = (pl.half + groups - 1) / groups;
    const uint32_t k0 = g * gs;
    uint32_t k1 = k0 + gs;
    if (k1 > pl.half) k1 = pl.half;
    ge_p3 run, tot;
    ge_identity(run);
    ge_identity(tot);
    for (uint32_t k = k1; k-- > k0;) {
        const uint32_t b = w * pl.half + k;
        if (offsets[b + 1] > offsets[b]) {
            ge_p3 p;
            kb_load_p3_w32(p, bucket_sum + 32 * (size_t)b);
            ge_cached pc;
            ge_to_cached(pc, p);
            ge_add<true>(run, run, pc);
        }
        ge_cached rc;
        ge_to_cached(rc, run);
        ge_add<true>(tot, tot, rc);
    }
    kb_store_p3_w32(part_run + 32 * tid, run);
    kb_store_p3_w32(part_tot + 32 * tid, tot);
}
// one thread's share of a window: groups [c0, c1) -> t1 = sum tot_g, t2 = sum g * run_g
KB_FN void kb_msm_window_chunk(ge_p3& t1, ge_p3& t2, uint32_t c0, uint32_t c1, const uint32_t* run_w, const uint32_t* tot_w)
{
    ge_p3 r, ws;
    ge_identity(r);
    ge_identity(ws);
    ge_identity(t1);
    for (uint32_t g = c1; g-- > c0;) {
        ge_p3 p;
        ge_cached pc;
        kb_load_p3_w32(p, run_w + 32 * (size_t)g);
        ge_to_cached(pc, p);
        ge_add<true>(r, r, pc);
        ge_to_cached(pc, r);
        ge_add<true>(ws, ws, pc);     // ws = sum (g - c0 + 1) run_g
        kb_load_p3_w32(p, tot_w + 32 * (size_t)g);
        ge_to_cached(pc, p);
        ge_add<true>(t1, t1, pc);
    }
    // sum g * run_g = ws + (c0 - 1) * r
    if (c0 >= 2 && c0 < c1) {
        ge_cached wc;
        ge_to_cached(wc, ws);
        kb_horner_step(r, (uint64_t)(c0 - 1), wc);
        t2 = r;
    } else if (c0 == 0 && c0 < c1) {
        // weights (g + 1): subtract one r
        ge_cached rc;
        ge_to_cached(rc, r);
        ge_addsub_rt(t2, ws, rc, true, true);
    } else {
        t2 = ws;
    }
}

#if !defined(KB_HOST_EMU)
// ======================================================================================
// kernels
// ======================================================================================
#if defined(KB_K_MSM)
// prepare + histogram in one pass: the digits are counted while the scalar is still at hand (counts zeroed by the caller)
static __global__ void __launch_bounds__(KB_THREADS) k_msm_prepare(kb_msm_plan pl, const uint8_t* points, const uint8_t* scalars, uint32_t* pts, uint32_t* mags, uint8_t* negs, uint32_t* bad, uint32_t* counts)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pl.n) return;
    uint32_t pw[8], sw[8];
    kb_load32(pw, points, i);   // coalesced 128-bit loads of the 32-byte encodings
    kb_load32(sw, scalars, i);
    kb_msm_prepare_body(i, pw, sw, pts, mags, negs, bad);
    kb_msm_hist_body(pl, i, mags, counts);
}
// The same for points that are already decoded: X, Y, Z, T as 4 x 8 words (any Z != 0) — what kb_point_decompress_batch,
// the MSM partials and every device-side producer of this library emit.  No 252-squaring decompression: one thread
// makes KB_INV_K points affine with ONE shared inversion (Montgomery's trick).  A point with Z = 0 or off the curve
// counts as bad and is replaced by the identity.
static __global__ void __launch_bounds__(KB_THREADS) k_msm_prepare_ext(kb_msm_plan pl, const uint32_t* points128, const uint8_t* scalars, uint32_t* pts, uint32_t* mags, uint8_t* negs, uint32_t* bad, uint32_t* counts)
{
    const size_t base = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * KB_INV_K;
    if (base >= pl.n) return;
    const int cnt = (pl.n - base < KB_INV_K) ? (int)(pl.n - base) : KB_INV_K;
    fe pref[KB_INV_K];
    fe acc, z, one;
    uint32_t zbad = 0;
    fe_set(one, 1);
    fe_set(acc, 1);
#pragma unroll 1
    for (int k = 0; k < cnt; k++) {
        kb_load_p3_z_w128(z, points128 + 32 * (base + k));
        const uint32_t z0 = fe_is_zero(z);
        zbad |= z0 << k;
        fe_cmov(z, one, z0);
        fe_mul(acc, acc, z);
        pref[k] = acc;
    }
    fe inv;
    fe_invert(inv, acc);
    const fe d = KB_FE_D, d2 = KB_FE_D2;
#pragma unroll 1
    for (int k = cnt - 1; k >= 0; k--) {
        const size_t i = base + k;
        fe zinv;
        kb_load_p3_z_w128(z, points128 + 32 * i);
        fe_cmov(z, one, (zbad >> k) & 1u);
        if (k > 0) {
            fe_mul(zinv, inv, pref[k - 1]);
            fe_mul(inv, inv, z);
        } else {
            zinv = inv;
        }
        fe x, y, xx, yy, l, r;
        kb_load_p3_xy_w128(x, y, points128 + 32 * i);
        fe_mul(x, x, zinv);
        fe_mul(y, y, zinv);
        // on the curve:  -x^2 + y^2 = 1 + d x^2 y^2
        fe_sq(xx, x);
        fe_sq(yy, y);
        fe_sub(l, yy, xx);
        fe_mul(r, xx, yy);
        fe_mul(r, r, d);
        fe_add(r, r, one);
        fe_sub(l, l, r);
        const uint32_t ok = fe_is_zero(l) & (((zbad >> k) & 1u) ^ 1u);
        ge_precomp q;
        fe_add(q.ypx, y, x);
        fe_sub(q.ymx, y, x);
        fe_mul(q.xy2d, x, y);
        fe_mul(q.xy2d, q.xy2d, d2);
        if (!ok) {
            ge_precomp_identity(q);
            atomicAdd(bad, 1u);
        }
        kb_store_precomp_w128(pts + 24 * i, q);
        uint32_t sw[8], mag[8], neg;
        kb_load32(sw, scalars, i);
        sc_effective(mag, neg, sw);
        kb_store32(reinterpret_cast<uint8_t*>(mags), i, mag);
        negs[i] = (uint8_t)neg;
        kb_msm_hist_body(pl, i, mags, counts);
    }
}
// exclusive scan of counts[0..nb) into offsets[0..nb], three launches:
//   tiles : each block scans a 2048-element tile (coalesced through shared memory), emits its total
//   sums  : one block scans the tile totals (<= 2048 tiles) and writes offsets[nb]
//   add   : adds each tile's base; clears cursor
#define KB_SCAN_TILE 2048
static __global__ void __launch_bounds__(256) k_msm_scan_tiles(uint32_t nb, const uint32_t* counts, uint32_t* offsets, uint32_t* tile_sums)
{
    __shared__ uint32_t buf[KB_SCAN_TILE];
    __shared__ uint32_t wsum[8];
    const uint32_t tid = threadIdx.x, base = blockIdx.x * KB_SCAN_TILE;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint32_t i = base + tid + 256 * k;
        buf[tid + 256 * k] = (i < nb) ? counts[i] : 0u;
    }
    __syncthreads();
    uint32_t v[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        v[k] = sum;
        sum += buf[8 * tid + k];
    }
    // exclusive scan of the 256 per-thread sums: warp shuffles, then the 8 warp totals
    uint32_t inc = sum;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t n = __shfl_up_sync(0xffffffffu, inc, off);
        if ((tid & 31) >= (uint32_t)off) inc += n;
    }
    if ((tid & 31) == 31) wsum[tid >> 5] = inc;
    __syncthreads();
    uint32_t wbase = 0;
    for (uint32_t w = 0; w < (tid >> 5); w++) wbase += wsum[w];
    const uint32_t excl = wbase + inc - sum;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 8; k++) buf[8 * tid + k] = excl + v[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint32_t i = base + tid + 256 * k;
        if (i < nb) offsets[i] = buf[tid + 256 * k];
    }
    if (tid == 255) tile_sums[blockIdx.x] = excl + sum;
}
static __global__ void __launch_bounds__(1024) k_msm_scan_sums(uint32_t ntiles, uint32_t nb, uint32_t* tile_sums, uint32_t* offsets)
{
    __shared__ uint32_t part[1024];
    const uint32_t tid = threadIdx.x;
    // each thread owns two consecutive tiles (ntiles <= 2048)
    const uint32_t a = (2 * tid < ntiles) ? tile_sums[2 * tid] : 0u;
    const uint32_t b = (2 * tid + 1 < ntiles) ? tile_sums[2 * tid + 1] : 0u;
    part[tid] = a + b;
    __syncthreads();
    for (uint32_t off = 1; off < 1024; off <<= 1) {
        const uint32_t v = (tid >= off) ? part[tid - off] : 0u;
        __syncthreads();
        part[tid] += v;
        __syncthreads();
    }
    const uint32_t excl = part[tid] - (a + b);
    if (2 * tid < ntiles) tile_sums[2 * tid] = excl;
    if (2 * tid + 1 < ntiles) tile_sums[2 * tid + 1] = excl + a;
    if (tid == 1023) offsets[nb] = part[1023];
}
static __global__ void __launch_bounds__(256) k_msm_scan_add(uint32_t nb, const uint32_t* tile_sums, uint32_t* offsets, uint32_t* cursor)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb) return;
    offsets[i] += tile_sums[i / KB_SCAN_TILE];
    cursor[i] = 0;
}
static __global__ void __launch_bounds__(256) k_msm_scatter(kb_msm_plan pl, const uint32_t* mags, const uint8_t* negs, const uint32_t* offsets, uint32_t* cursor, uint32_t* sorted)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pl.n) return;
    kb_msm_scatter_body(pl, i, mags, negs, offsets, cursor, sorted);
}
static __global__ void __launch_bounds__(KB_THREADS) k_msm_accum(kb_msm_plan pl, size_t nthreads, const uint32_t* offsets, const uint32_t* sorted, const uint32_t* pts, uint32_t* bucket_sum, uint32_t* heads,
                                                          uint32_t* tails, uint8_t* flags, uint32_t* tailb)
{
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nthreads) return;
    kb_msm_accum_body(pl, t, offsets, sorted, pts, bucket_sum, heads, tails, flags, tailb);
}
static __global__ void __launch_bounds__(KB_THREADS) k_msm_merge(kb_msm_plan pl, size_t nthreads, const uint32_t* offsets, uint32_t* long_count, uint32_t* long_list, uint32_t* bucket_sum,
                                                          const uint32_t* heads, const uint32_t* tails, const uint8_t* flags, const uint32_t* tailb, int mode)
{
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nthreads) return;
    kb_msm_merge_body(pl, t, nthreads, offsets, 8u, long_count, long_list, bucket_sum, heads, tails, flags, tailb, mode);
}
static __global__ void __launch_bounds__(KB_THREADS) k_msm_reduce(kb_msm_plan pl, uint32_t groups, const uint32_t* offsets, const uint32_t* bucket_sum, uint32_t* part_run, uint32_t* part_tot)
{
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= (size_t)pl.windows * groups) return;
    kb_msm_reduce_body(pl, tid, groups, offsets, bucket_sum, part_run, part_tot);
}

#endif  // KB_K_MSM (first part)
// butterfly sum of one point per lane: after the call every lane holds the warp total
__device__ __forceinline__ void kb_warp_sum_point(ge_p3& p)
{
#pragma unroll 1
    for (int off = 16; off >= 1; off >>= 1) {
        ge_p3 q;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            q.X.v[k] = __shfl_xor_sync(0xffffffffu, p.X.v[k], off);
            q.Y.v[k] = __shfl_xor_sync(0xffffffffu, p.Y.v[k], off);
            q.Z.v[k] = __shfl_xor_sync(0xffffffffu, p.Z.v[k], off);
            q.T.v[k] = __shfl_xor_sync(0xffffffffu, p.T.v[k], off);
        }
        ge_cached qc;
        ge_to_cached(qc, q);
        ge_add<true>(p, p, qc);
    }
}
// two independent butterflies in one loop: the additions of a level do not depend on each other, so a warp that runs
// alone on its scheduler (the folds at the end of an MSM) overlaps their latencies
__device__ __forceinline__ void kb_warp_sum_point2(ge_p3& p, ge_p3& r)
{
#pragma unroll 1
    for (int off = 16; off >= 1; off >>= 1) {
        ge_p3 q, u;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            q.X.v[k] = __shfl_xor_sync(0xffffffffu, p.X.v[k], off);
            q.Y.v[k] = __shfl_xor_sync(0xffffffffu, p.Y.v[k], off);
            q.Z.v[k] = __shfl_xor_sync(0xffffffffu, p.Z.v[k], off);
            q.T.v[k] = __shfl_xor_sync(0xffffffffu, p.T.v[k], off);
            u.X.v[k] = __shfl_xor_sync(0xffffffffu, r.X.v[k], off);
            u.Y.v[k] = __shfl_xor_sync(0xffffffffu, r.Y.v[k], off);
            u.Z.v[k] = __shfl_xor_sync(0xffffffffu, r.Z.v[k], off);
            u.T.v[k] = __shfl_xor_sync(0xffffffffu, r.T.v[k], off);
        }
        ge_cached qc, uc;
        ge_to_cached(qc, q);
        ge_to_cached(uc, u);
        ge_add<true>(p, p, qc);
        ge_add<true>(r, r, uc);
    }
}
#if defined(KB_K_MSM)
// long runs: one BLOCK per queued (t, u_end, bucket): its threads stride over the head partials of chunks t+1 .. u_end-1,
// sum them by warp butterflies and across the warps through shared memory; thread 0 adds tail[t] and owns the bucket.
// (A run of thousands of chunks — the top window of reduced scalars holds a single bucket — used to be one warp's work.)
#define KB_MSM_LONG_THREADS 256
static __global__ void __launch_bounds__(KB_MSM_LONG_THREADS) k_msm_merge_long(size_t nthreads, const uint32_t* long_count, const uint32_t* long_list, uint32_t* bucket_sum, const uint32_t* heads,
                                                                                 const uint32_t* tails, const uint8_t* flags)
{
    __shared__ uint32_t wsum[(KB_MSM_LONG_THREADS / 32) * 32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t count = *long_count;
    for (uint32_t e = blockIdx.x; e < count; e += gridDim.x) {
        const size_t t = long_list[3 * e];
        size_t u_end = long_list[3 * e + 1];
        if (u_end > nthreads) u_end = nthreads;
        const uint32_t b = long_list[3 * e + 2];
        ge_p3 s;
        ge_identity(s);
        for (size_t u = t + 1 + threadIdx.x; u < u_end; u += KB_MSM_LONG_THREADS) {
            if (flags[u] & 1u) {
                ge_p3 h;
                kb_load_p3_w32(h, heads + 32 * u);
                ge_cached hc;
                ge_to_cached(hc, h);
                ge_add<true>(s, s, hc);
            }
        }
        kb_warp_sum_point(s);
        __syncthreads();   // the previous entry's readers are done with wsum
        if (lane == 0) kb_store_p3_w32(wsum + 32 * warp, s);
        __syncthreads();
        if (warp == 0) {
            ge_identity(s);
            if (lane < KB_MSM_LONG_THREADS / 32) kb_load_p3_w32(s, wsum + 32 * lane);
            kb_warp_sum_point(s);
            if (lane == 0) {
                ge_p3 tl;
                kb_load_p3_w32(tl, tails + 32 * t);
                ge_cached tc;
                ge_to_cached(tc, tl);
                ge_add<true>(s, s, tc);
                kb_store_p3_w32(bucket_sum + 32 * (size_t)b, s);
            }
        }
    }
}
// window sums: block w folds the group partials of window w:  S_w = sum_g tot_g + gs * sum_g g * run_g.
// Each of the 256 threads owns a contiguous run of groups (kb_msm_window_chunk), the two partial points are summed
// with a warp-shuffle butterfly and then across the 8 warps through shared memory.
static __global__ void __launch_bounds__(256) k_msm_window_sums(kb_msm_plan pl, uint32_t groups, const uint32_t* part_run, const uint32_t* part_tot, uint32_t* win_sum)
{
    __shared__ uint32_t wtot[2 * 8 * 32];
    const uint32_t w = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t per = (groups + blockDim.x - 1) / blockDim.x;
    uint32_t c0 = threadIdx.x * per, c1 = c0 + per;
    if (c0 > groups) c0 = groups;
    if (c1 > groups) c1 = groups;
    ge_p3 t1, t2;
    kb_msm_window_chunk(t1, t2, c0, c1, part_run + 32 * (size_t)w * groups, part_tot + 32 * (size_t)w * groups);
    kb_warp_sum_point2(t1, t2);
    if (lane == 0) {
        kb_store_p3_w32(wtot + 32 * warp, t1);
        kb_store_p3_w32(wtot + 32 * (8 + warp), t2);
    }
    __syncthreads();
    if (warp == 0) {
        ge_p3 a, b;
        ge_identity(a);
        ge_identity(b);
        if (lane < 8) {
            kb_load_p3_w32(a, wtot + 32 * lane);
            kb_load_p3_w32(b, wtot + 32 * (8 + lane));
        }
        kb_warp_sum_point2(a, b);
        if (lane == 0) {
            const uint32_t gs = (pl.half + groups - 1) / groups;
            ge_cached ac;
            ge_to_cached(ac, a);
            kb_horner_step(b, (uint64_t)gs, ac);   // b = gs * b + a
            kb_store_p3_w32(win_sum + 32 * w, b);
        }
    }
}
// One doubling shared by 4 adjacent lanes: the four squarings (X^2, Y^2, Z^2, (X+Y)^2) and then the four
// products (E*F, G*H, F*G, E*H) of the doubling formula are independent, so each lane of a quad does ONE of
// them and the results travel by warp shuffle.  The chain of ~270 dependent doublings that closes an MSM
// (Horner over the windows) is pure latency for a single thread; this cuts it about three-fold.
// Every lane of the quad enters with the same point and leaves with the same doubled point.
__device__ __forceinline__ void kb_shfl_fe(fe& out, const fe& in, int src_lane)
{
#pragma unroll
    for (int k = 0; k < 8; k++) out.v[k] = __shfl_sync(0xffffffffu, in.v[k], src_lane);
}
__device__ __forceinline__ void kb_dbl_quad(ge_p3& p)
{
    const int lane = threadIdx.x & 31, role = lane & 3, base = lane & ~3;
    fe in = p.X, t, sq;
    fe_add(t, p.X, p.Y);
    fe_cmov(in, p.Y, (uint32_t)(role == 1));
    fe_cmov(in, p.Z, (uint32_t)(role == 2));
    fe_cmov(in, t, (uint32_t)(role == 3));
    fe_sq(sq, in);
    fe a, b, c, d, e, f, g, h;
    kb_shfl_fe(a, sq, base + 0);
    kb_shfl_fe(b, sq, base + 1);
    kb_shfl_fe(c, sq, base + 2);
    kb_shfl_fe(d, sq, base + 3);
    fe_dbl(c, c);
    fe_add(h, a, b);
    fe_sub(e, h, d);
    fe_sub(g, a, b);
    fe_add(f, c, g);
    // role 0: E*F   1: G*H   2: F*G   3: E*H
    fe l = e, r = f, prod;
    fe_cmov(l, g, (uint32_t)(role == 1));
    fe_cmov(l, f, (uint32_t)(role == 2));
    fe_cmov(r, h, (uint32_t)(role == 1 || role == 3));
    fe_cmov(r, g, (uint32_t)(role == 2));
    fe_mul(prod, l, r);
    kb_shfl_fe(p.X, prod, base + 0);
    kb_shfl_fe(p.Y, prod, base + 1);
    kb_shfl_fe(p.Z, prod, base + 2);
    kb_shfl_fe(p.T, prod, base + 3);
}
// finish: Horner over the windows (c quad-doublings per window), add to the running total `acc128`
// (X,Y,Z,T words) and, if out32 != nullptr, write its encoding.  One warp; all quads compute the same thing.
static __global__ void k_msm_finish(kb_msm_plan pl, const uint32_t* win_sum, uint32_t* acc128, int first_chunk, uint8_t* out32)
{
    if (blockIdx.x != 0 || threadIdx.x >= 32) return;
    ge_p3 tot;
    ge_identity(tot);
    for (uint32_t w = pl.windows; w-- > 0;) {
        for (uint32_t k = 0; k < pl.c; k++) kb_dbl_quad(tot);
        ge_p3 s;
        kb_load_p3_w32(s, win_sum + 32 * w);
        ge_cached sc;
        ge_to_cached(sc, s);
        ge_add<true>(tot, tot, sc);
    }
    if (!first_chunk) {
        ge_p3 prev;
        kb_load_p3_w32(prev, acc128);
        ge_cached pc;
        ge_to_cached(pc, prev);
        ge_add<true>(tot, tot, pc);
    }
    __syncwarp();
    if (threadIdx.x != 0) return;
    kb_store_p3_w32(acc128, tot);
    if (out32) {
        uint32_t o[8];
        ge_compress(o, tot);
        kb_store32(out32, 0, o);
    }
}
#endif  // KB_K_MSM (second part)
// out = compress(sum of k uncompressed partials): the fold after the cross-GPU gather
static __global__ void k_point_sum(size_t k, const uint32_t* partials, uint8_t* out32)
{
    const uint32_t lane = threadIdx.x & 31;
    ge_p3 s;
    ge_identity(s);
    for (size_t g = lane; g < k; g += 32) {
        ge_p3 p;
        kb_load_p3_w32(p, partials + 32 * g);
        ge_cached pc;
        ge_to_cached(pc, p);
        ge_add<true>(s, s, pc);
    }
    kb_warp_sum_point(s);
    if (lane == 0) {
        uint32_t o[8];
        ge_compress(o, s);
        kb_store32(out32, 0, o);
    }
}

// Column sums of npoly committed polynomials: out[j] = sum_d commits[d][j] — the repeated PubPoly::add of
// dkg_key (share/dkg/pedersen/dkg.rs:905-954, share/poly.rs:486-509).  One warp per coefficient: lanes
// stride over the dealers (cached operand form from k_commit_prepare), shuffle butterfly, lane 0 stores.
static __global__ void __launch_bounds__(KB_THREADS) k_poly_colsum(size_t npoly, size_t t, const uint32_t* cached, const uint8_t* bad, uint32_t* xyz, uint8_t* status)
{
    const uint32_t lane = threadIdx.x & 31;
    const size_t j = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= t) return;
    ge_p3 s;
    ge_identity(s);
    uint32_t anybad = 0;
    for (size_t d = lane; d < npoly; d += 32) {
        ge_cached c;
        kb_load_cached_w128(c, cached + 32 * (d * t + j));
        anybad |= bad[d * t + j];
        ge_add<true>(s, s, c);
    }
    kb_warp_sum_point(s);
    anybad = __any_sync(0xffffffffu, anybad != 0);
    if (lane == 0) {
        if (anybad) ge_identity(s);
        kb_store_xyz(xyz, j, s);
        status[j] = (uint8_t)anybad;
    }
}

#endif  // !KB_HOST_EMU
