// capi_msm.cu — Pippenger multi-scalar multiplication entry points (msm.cuh)
#define KB_K_MSM
#include "ctx.cuh"
#include "kernels.cuh"
#include "msm.cuh"
// ------------------------------------------------------------------------------------
// Pippenger driver (msm.cuh): chunks of <= KB_MSM_CHUNK points, partial sums chained on device
// ------------------------------------------------------------------------------------
int kb_msm_run(kb_ctx* ctx, size_t n, const uint8_t* d_scalars, const void* d_points, int ext, uint8_t* d_out32, uint32_t* d_partial128, unsigned long long* d_bad, cudaStream_t st)
{
    uint32_t* acc128 = d_partial128;
    if (!acc128) KB_SCRATCH(10, 128, acc128);
    uint32_t* bad;
    if (d_bad) bad = reinterpret_cast<uint32_t*>(d_bad);
    else KB_SCRATCH(11, 8, bad);
    KB_CUDA(cudaMemsetAsync(bad, 0, 8, st));
    if (n == 0) {
        kb_msm_plan pl = {0, 4, 0, 8, 0, 16};
        k_msm_finish<<<1, 32, 0, st>>>(pl, nullptr, acc128, 1, d_out32);
        KB_LAUNCHED();
        return KB_OK;
    }
    for (size_t off = 0; off < n; off += KB_MSM_CHUNK) {
        const size_t cn = (n - off < KB_MSM_CHUNK) ? (n - off) : KB_MSM_CHUNK;
        kb_msm_plan pl;
        pl.n = (uint32_t)cn;
        pl.c = kb_msm_window_bits_host(cn);
        if (ctx->msm_c) pl.c = (uint32_t)ctx->msm_c;   // KB_MSM_C tuning override; measured at 2^22: c = 15 / 16 / 17 -> 15.6 / 15.3 / 15.6 ms
        pl.windows = (257 + pl.c - 1) / pl.c;
        pl.half = 1u << (pl.c - 1);
        pl.nb = pl.windows * pl.half;
        pl.k = kb_msm_chunk_entries(cn, pl.half);
        const uint32_t groups = kb_msm_groups_host(pl.half, (uint32_t)ctx->msm_groups);
        const size_t nthreads = (cn * pl.windows + pl.k - 1) / pl.k;
        uint32_t *pts, *mags, *counts, *offsets, *cursor, *sorted, *bucket_sum, *heads, *tails, *partial, *tile_sums, *long_list, *win_sum;
        uint8_t *negs, *flags;
        uint32_t* tailb;
        KB_SCRATCH(12, 96 * cn, pts);
        KB_SCRATCH(13, 32 * cn, mags);
        KB_SCRATCH(14, cn, negs);
        KB_SCRATCH(15, 4 * (size_t)pl.nb, counts);
        KB_SCRATCH(16, 4 * ((size_t)pl.nb + 1), offsets);
        KB_SCRATCH(17, 4 * (size_t)pl.nb, cursor);
        KB_SCRATCH(18, 4 * cn * pl.windows, sorted);
        KB_SCRATCH(19, 128 * (size_t)pl.nb, bucket_sum);
        KB_SCRATCH(20, 128 * nthreads, heads);
        KB_SCRATCH(21, 128 * nthreads, tails);
        KB_SCRATCH(22, nthreads, flags);
        KB_SCRATCH(53, 4 * nthreads, tailb);
        KB_SCRATCH(23, 2 * 128 * (size_t)pl.windows * groups, partial);
        uint32_t* part_tot = partial + 32 * (size_t)pl.windows * groups;
        KB_SCRATCH(24, 4 * 2048, tile_sums);
        KB_SCRATCH(25, 16 + 12 * (size_t)pl.nb, long_list);  // at most one long run per bucket
        KB_SCRATCH(26, 128 * (size_t)pl.windows, win_sum);
        if (pl.nb > 2048u * KB_SCAN_TILE) return KB_ERR_ARG;
        KB_CUDA(cudaMemsetAsync(counts, 0, 4 * (size_t)pl.nb, st));
        // decode (or, for points that are already decoded, make affine with shared inversions) + digit histogram
        if (ext) k_msm_prepare_ext<<<kb_blocks((cn + KB_INV_K - 1) / KB_INV_K, KB_THREADS), KB_THREADS, 0, st>>>(pl, (const uint32_t*)d_points + 32 * off, d_scalars + 32 * off, pts, mags, negs, bad, counts);
        else k_msm_prepare<<<kb_blocks(cn, KB_THREADS), KB_THREADS, 0, st>>>(pl, (const uint8_t*)d_points + 32 * off, d_scalars + 32 * off, pts, mags, negs, bad, counts);
        KB_LAUNCHED();
        const uint32_t ntiles = (pl.nb + KB_SCAN_TILE - 1) / KB_SCAN_TILE;
        k_msm_scan_tiles<<<ntiles, 256, 0, st>>>(pl.nb, counts, offsets, tile_sums);
        KB_LAUNCHED();
        k_msm_scan_sums<<<1, 1024, 0, st>>>(ntiles, pl.nb, tile_sums, offsets);
        KB_LAUNCHED();
        k_msm_scan_add<<<kb_blocks(pl.nb, 256), 256, 0, st>>>(pl.nb, tile_sums, offsets, cursor);
        KB_LAUNCHED();
        k_msm_scatter<<<kb_blocks(cn, 256), 256, 0, st>>>(pl, mags, negs, offsets, cursor, sorted);
        KB_LAUNCHED();
        k_msm_accum<<<kb_blocks(nthreads, KB_THREADS), KB_THREADS, 0, st>>>(pl, nthreads, offsets, sorted, pts, bucket_sum, heads, tails, flags, tailb);
        KB_LAUNCHED();
        KB_CUDA(cudaMemsetAsync(long_list, 0, 4, st));  // word 0 of the block is the queue length
        // The long runs (few, summed by whole blocks) and the short ones (many, one thread each) touch different buckets:
        // a first pass only queues the long ones, then the two kernels run side by side on two streams.
        cudaStream_t side = (st == ctx->stream2) ? ctx->stream : ctx->stream2;
        k_msm_merge<<<kb_blocks(nthreads, KB_THREADS), KB_THREADS, 0, st>>>(pl, nthreads, offsets, long_list, long_list + 4, bucket_sum, heads, tails, flags, tailb, 1);
        KB_LAUNCHED();
        KB_CUDA(cudaEventRecord(ctx->fork_ev, st));
        KB_CUDA(cudaStreamWaitEvent(side, ctx->fork_ev, 0));
        k_msm_merge_long<<<ctx->sm_count * 2, KB_MSM_LONG_THREADS, 0, side>>>(nthreads, long_list, long_list + 4, bucket_sum, heads, tails, flags);
        KB_LAUNCHED();
        KB_CUDA(cudaEventRecord(ctx->join_ev, side));
        k_msm_merge<<<kb_blocks(nthreads, KB_THREADS), KB_THREADS, 0, st>>>(pl, nthreads, offsets, long_list, long_list + 4, bucket_sum, heads, tails, flags, tailb, 2);
        KB_LAUNCHED();
        KB_CUDA(cudaStreamWaitEvent(st, ctx->join_ev, 0));
        k_msm_reduce<<<kb_blocks((size_t)pl.windows * groups, KB_THREADS), KB_THREADS, 0, st>>>(pl, groups, offsets, bucket_sum, partial, part_tot);
        KB_LAUNCHED();
        k_msm_window_sums<<<pl.windows, 256, 0, st>>>(pl, groups, partial, part_tot, win_sum);
        KB_LAUNCHED();
        const bool last = off + cn >= n;
        k_msm_finish<<<1, 32, 0, st>>>(pl, win_sum, acc128, off == 0 ? 1 : 0, last ? d_out32 : nullptr);
        KB_LAUNCHED();
    }
    return KB_OK;
}

extern "C" {
// ------------------------------------------------------------------------------------
// MSM
// ------------------------------------------------------------------------------------
int kb_dev_msm(kb_ctx* ctx, size_t n, const void* d_scalars, const void* d_points, void* d_out32, void* d_partial128, void* d_bad_points, void* stream)
{
    if (!ctx || (n && (!d_scalars || !d_points)) || (!d_out32 && !d_partial128)) return KB_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    KB_DEV_RETURN(st, kb_msm_run(ctx, n, (const uint8_t*)d_scalars, d_points, 0, (uint8_t*)d_out32, (uint32_t*)d_partial128, (unsigned long long*)d_bad_points, st));
}
int kb_dev_msm_ext(kb_ctx* ctx, size_t n, const void* d_scalars, const void* d_points128, void* d_out32, void* d_partial128, void* d_bad_points, void* stream)
{
    if (!ctx || (n && (!d_scalars || !d_points128)) || (!d_out32 && !d_partial128)) return KB_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    KB_DEV_RETURN(st, kb_msm_run(ctx, n, (const uint8_t*)d_scalars, d_points128, 1, (uint8_t*)d_out32, (uint32_t*)d_partial128, (unsigned long long*)d_bad_points, st));
}
int kb_msm(kb_ctx* ctx, size_t n, const uint8_t* scalars, const uint8_t* points, uint8_t* out32, uint8_t* partial128, uint64_t* bad_points)
{
    KB_ENTER();
    if ((n && (!scalars || !points)) || (!out32 && !partial128)) return KB_ERR_ARG;
    uint8_t *d_s, *d_p, *d_o;
    KB_SCRATCH(0, 32 * n, d_s);
    KB_SCRATCH(2, 32 * n, d_p);
    KB_SCRATCH(1, 32 + 128 + 8, d_o);
    if (n) {
        KB_H2D(d_s, scalars, 32 * n);
        KB_H2D(d_p, points, 32 * n);
    }
    int rc = kb_dev_msm(ctx, n, d_s, d_p, d_o, d_o + 32, d_o + 160, ctx->stream);
    if (rc != KB_OK) return rc;
    if (out32) KB_D2H(out32, d_o, 32);
    if (partial128) KB_D2H(partial128, d_o + 32, 128);
    if (bad_points) KB_D2H(bad_points, d_o + 160, 8);
    KB_SYNC();
    return KB_OK;
}
int kb_dev_point_sum(kb_ctx* ctx, size_t k, const void* d_partials128, void* d_out32, void* stream)
{
    if (!ctx || !d_out32 || (k && !d_partials128)) return KB_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    k_point_sum<<<1, 32, 0, st>>>(k, (const uint32_t*)d_partials128, (uint8_t*)d_out32);
    KB_LAUNCHED();
    KB_DEV_RETURN(st, KB_OK);
}
int kb_point_sum(kb_ctx* ctx, size_t k, const uint8_t* partials128, uint8_t* out32)
{
    KB_ENTER();
    if (!out32 || (k && !partials128)) return KB_ERR_ARG;
    uint8_t *d_i, *d_o;
    KB_SCRATCH(0, 128 * k, d_i);
    KB_SCRATCH(1, 32, d_o);
    if (k) KB_H2D(d_i, partials128, 128 * k);
    int rc = kb_dev_point_sum(ctx, k, d_i, d_o, ctx->stream);
    if (rc != KB_OK) return rc;
    KB_D2H(out32, d_o, 32);
    KB_SYNC();
    return KB_OK;
}

}  // extern "C"
