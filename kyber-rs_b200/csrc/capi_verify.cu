// capi_verify.cu — eddsa::verify_with_checks / schnorr::verify_with_checks and EdDSA::sign entry points
#define KB_K_SIGN
// Field-arithmetic bodies of THIS translation unit (fe.cuh): the zero-free row order of fe_mul / fe_sq and the borrow-mask
// wrap of fe_sub.  All bodies are bit-exact; which one is faster depends on the kernel (the balance ptxas strikes between
// the ALU and the multiplier pipe).  Measured, round 2, one B200: the verify step gains 0.8 % with all three
// (k_verify_half_main 16.54 -> 16.42 ms, k_verify_half_prep 4.96 -> 4.90 ms) while the MSM and DKG kernels lose 1-4 %,
// so only the verifiers (and the signing kernels that share this unit) are built with them.
#define KB_FE_MUL_RIP
#define KB_FE_SQ_RIP
#define KB_FE_SUBMASK
#include "ctx.cuh"
#include "kernels.cuh"
int kb_verify_launch(kb_ctx* ctx, size_t n, const uint8_t* d_pk, const uint8_t* d_msg, const uint64_t* d_msg_off, uint64_t msg_base, const uint8_t* d_sig, uint8_t* d_status, int schnorr,
                            uint32_t* xyz, uint8_t* fl, cudaStream_t st)
{
    const unsigned th = kb_item_threads(ctx, n);
    const unsigned g1 = kb_blocks(n, th), g2 = kb_blocks((n + KB_INV_K - 1) / KB_INV_K, KB_THREADS);
    const bool tm = ctx->timing != 0;
    if (!ctx->verify_full) {
        // the 96-byte-per-item xyz scratch of the full-length path is not needed; `xyz` carries the records
        const unsigned gp = kb_blocks(n, KB_THREADS);
        if (tm) cudaEventRecord(ctx->tev[0], st);
        if (ctx->verify_split == 2 || (ctx->verify_split && n >= (size_t)ctx->sm_count * KB_THREADS)) {   // 2: every batch size (tests)
            // two kernels side by side (kernels.cuh): the persistent scalars kernel first, on the side stream of this lane
            const int lane = (st == ctx->stream2) ? 1 : 0;
            cudaStream_t side = ctx->vs_side[lane];
            unsigned long long* counter = ctx->vs_counter + lane;
            const unsigned gs = (unsigned)(ctx->sm_count * ctx->vs_blocks);
            KB_CUDA(cudaEventRecord(ctx->vs_fork[lane], st));
            KB_CUDA(cudaStreamWaitEvent(side, ctx->vs_fork[lane], 0));
            KB_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), side));
            if (schnorr) k_verify_half_scalars<true><<<gs, KB_THREADS, 0, side>>>(n, d_pk, d_msg, d_msg_off, msg_base, d_sig, xyz, counter);
            else k_verify_half_scalars<false><<<gs, KB_THREADS, 0, side>>>(n, d_pk, d_msg, d_msg_off, msg_base, d_sig, xyz, counter);
            KB_LAUNCHED();
            KB_CUDA(cudaEventRecord(ctx->vs_join[lane], side));
            if (ctx->vs_pbound == 4) k_verify_half_points<4><<<gp, KB_THREADS, 0, st>>>(n, d_pk, d_sig, xyz);
            else if (ctx->vs_pbound == 6) k_verify_half_points<6><<<gp, KB_THREADS, 0, st>>>(n, d_pk, d_sig, xyz);
            else k_verify_half_points<5><<<gp, KB_THREADS, 0, st>>>(n, d_pk, d_sig, xyz);
            KB_LAUNCHED();
            KB_CUDA(cudaStreamWaitEvent(st, ctx->vs_join[lane], 0));
            if (schnorr) k_verify_half_fix<true><<<kb_blocks(n, 256), 256, 0, st>>>(n, xyz);
            else k_verify_half_fix<false><<<kb_blocks(n, 256), 256, 0, st>>>(n, xyz);
            KB_LAUNCHED();
        } else {
            if (schnorr) k_verify_half_prep<true><<<gp, KB_THREADS, 0, st>>>(n, d_pk, d_msg, d_msg_off, msg_base, d_sig, xyz);
            else k_verify_half_prep<false><<<gp, KB_THREADS, 0, st>>>(n, d_pk, d_msg, d_msg_off, msg_base, d_sig, xyz);
            KB_LAUNCHED();
        }
        if (tm) cudaEventRecord(ctx->tev[1], st);
        // Records sorted by the length of their loop (kernels.cuh k_half_sort_*): the trip count of the main kernel is
        // uniform over a block, so a block of like records stops at ITS length instead of the longest of 128 random ones.
        const uint32_t* perm = nullptr;
#if KB_HALF_JOINT
        if (ctx->verify_sort && (n >= 16384 || ctx->verify_sort == 2) && n < ((size_t)1 << 32)) {   // 2: every batch size (tests)
            uint32_t* pm = reinterpret_cast<uint32_t*>(fl);
            uint8_t* keys = fl + 4 * n;
            uint32_t* hist = reinterpret_cast<uint32_t*>(fl + ((5 * n + 255) & ~(size_t)255));
            KB_CUDA(cudaMemsetAsync(hist, 0, 4 * KB_SORT_BINS, st));
            k_half_sort_count<<<kb_blocks(n, 256), 256, 0, st>>>(n, xyz, keys, hist);
            KB_LAUNCHED();
            k_half_sort_scan<<<1, 32, 0, st>>>(hist, hist + KB_SORT_BINS);
            KB_LAUNCHED();
            k_half_sort_scatter<<<kb_blocks(n, 256), 256, 0, st>>>(n, keys, hist + KB_SORT_BINS, pm);
            KB_LAUNCHED();
            perm = pm;
        }
#endif
        if (schnorr) k_verify_half_main<true><<<g1, th, 0, st>>>(n, xyz, perm, d_status, ctx->comb, ctx->verify_min_windows);
        else k_verify_half_main<false><<<g1, th, 0, st>>>(n, xyz, perm, d_status, ctx->comb, ctx->verify_min_windows);
        KB_LAUNCHED();
        if (tm) {
            cudaEventRecord(ctx->tev[2], st);
            ctx->timing_valid = 1;
        }
        return KB_OK;
    }
    if (tm) cudaEventRecord(ctx->tev[0], st);
    if (schnorr) k_verify_stage1<true><<<g1, th, 0, st>>>(n, d_pk, d_msg, d_msg_off, msg_base, d_sig, xyz, fl, ctx->base128);
    else k_verify_stage1<false><<<g1, th, 0, st>>>(n, d_pk, d_msg, d_msg_off, msg_base, d_sig, xyz, fl, ctx->base128);
    KB_LAUNCHED();
    if (tm) cudaEventRecord(ctx->tev[1], st);
    if (schnorr) k_verify_stage2<true><<<g2, KB_THREADS, 0, st>>>(n, xyz, fl, d_sig, d_status);
    else k_verify_stage2<false><<<g2, KB_THREADS, 0, st>>>(n, xyz, fl, d_sig, d_status);
    KB_LAUNCHED();
    if (tm) {
        cudaEventRecord(ctx->tev[2], st);
        ctx->timing_valid = 1;
    }
    return KB_OK;
}

extern "C" {
int kb_dev_eddsa_verify(kb_ctx* ctx, size_t n, const void* d_pk, const void* d_msg, const void* d_msg_off, const void* d_sig, void* d_status, int schnorr, void* stream)
{
    if (!ctx || (n && (!d_pk || !d_msg_off || !d_sig || !d_status))) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    uint32_t* xyz;
    uint8_t* fl;
    KB_SCRATCH(KB_SLOT_XYZ, KB_VERIFY_SCRATCH_BYTES * n, xyz);
    KB_SCRATCH(KB_SLOT_FLAGS, KB_VERIFY_FLAG_BYTES(n), fl);
    KB_DEV_RETURN(st, kb_verify_launch(ctx, n, (const uint8_t*)d_pk, (const uint8_t*)d_msg, (const uint64_t*)d_msg_off, 0, (const uint8_t*)d_sig, (uint8_t*)d_status, schnorr, xyz, fl, st));
}
// Host-buffer verification, pipelined: the batch is cut into chunks that alternate between two staging lanes, so the
// H2D copy of chunk k+1 and the D2H of chunk k-1 overlap the kernels of chunk k (each lane owns its own staging and
// scratch buffers).
#define KB_VERIFY_MAX_CHUNKS 4096
static int kb_verify_host(kb_ctx* ctx, size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status, int schnorr)
{
    KB_ENTER();
    if (n && (!pk || !msg_off || !sig || !status)) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    if (msg_off[n] && !msg) return KB_ERR_ARG;
    // Chunk sizes.  Measured on a 2^20 batch (tools/e2e_sweep.py, round 2): whole WAVES of the main kernel — its resident
    // blocks of 128 signatures per SM: 56 832 signatures on 148 SMs at the 3 blocks of that measurement, 75 776 at today's 4 —
    // beat powers of two, and the chunks GROW: a third of
    // a wave first (the kernels start after a copy of 3 MB), then four times the previous chunk each, up to the cap.  A
    // chunk's copy (168 B per signature at PCIe speed) is shorter than the kernels of the chunk before it as long as the
    // growth factor stays below about 6, so the device never waits for a copy after the first one, and a 2^20 batch is
    // 4 chunks (8 launches) instead of 6.
    const size_t wave = (size_t)ctx->sm_count * KB_VERIFY_HALF_MINBLOCKS * KB_THREADS;
    size_t cap = ctx->verify_chunk_n ? ctx->verify_chunk_n : ctx->verify_chunk;
    if (cap == 0) cap = 16 * wave;
    // cut[k] .. cut[k+1]: signatures of chunk k
    size_t cut[KB_VERIFY_MAX_CHUNKS + 1];
    size_t nchunks = 0;
    cut[0] = 0;
    {
        size_t lo = 0, step = wave / 3;
        if (step > cap) step = cap;
        while (lo < n) {
            if (nchunks + 1 == KB_VERIFY_MAX_CHUNKS) step = n - lo;   // (never with the default sizes: 2^35 signatures)
            lo = (lo + step < n) ? lo + step : n;
            cut[++nchunks] = lo;
            step = (step == wave / 3) ? wave : 4 * step;
            if (step > cap) step = cap;
        }
    }
    size_t max_mbytes = 0, cn_max = 0;
    for (size_t k = 0; k < nchunks; k++) {
        if (msg_off[cut[k + 1]] < msg_off[cut[k]]) return KB_ERR_ARG;
        const size_t mb = (size_t)(msg_off[cut[k + 1]] - msg_off[cut[k]]);
        if (mb > max_mbytes) max_mbytes = mb;
        if (cut[k + 1] - cut[k] > cn_max) cn_max = cut[k + 1] - cut[k];
    }
    cudaStream_t lane[2] = {ctx->stream, ctx->stream2};
    uint8_t *d_pk[2], *d_sig[2], *d_m[2], *d_st[2], *fl[2];
    uint64_t* d_off[2];
    uint32_t* xyz[2];
    for (int l = 0; l < 2; l++) {
        const int b = 32 + 7 * l;
        KB_SCRATCH(b + 0, 32 * cn_max, d_pk[l]);
        KB_SCRATCH(b + 1, 64 * cn_max, d_sig[l]);
        KB_SCRATCH(b + 2, max_mbytes, d_m[l]);
        KB_SCRATCH(b + 3, 8 * (cn_max + 1), d_off[l]);
        KB_SCRATCH(b + 4, cn_max, d_st[l]);
        KB_SCRATCH(b + 5, KB_VERIFY_SCRATCH_BYTES * cn_max, xyz[l]);
        KB_SCRATCH(b + 6, KB_VERIFY_FLAG_BYTES(cn_max), fl[l]);
    }
    // Two schedules.  verify_pipe = 0 (default): two independent lanes (copy in, kernels, copy out each) that alternate;
    // the device may run the kernels of consecutive chunks side by side, which fills the tail of every launch.
    // verify_pipe = 1: the kernels of ALL chunks on one stream, in order, the copies on the other one, tied together by
    // events per staging lane — the preparation of chunk k+1 then never shares an SM with the main loop of chunk k.
    // Measured (tools/e2e_sweep.py): 47.1 M sigs/s at best against 47.7 M for the two lanes — the filled tails are worth
    // more than the undisturbed instruction cache.
    const bool pipe = ctx->verify_pipe != 0;
    cudaStream_t compute = ctx->stream, copy = ctx->stream2;
    for (size_t k = 0; k < nchunks; k++) {
        const int l = (int)(k & 1);
        const size_t lo = cut[k], hi = cut[k + 1], cn = hi - lo;
        // the offsets of a chunk are validated right before it is enqueued: the walk over the next chunk's offsets then
        // runs while the device works on this one (a kernel that met hi < lo would read out of bounds)
        if (!kb_msg_off_ok(cn, msg_off + lo)) {
            cudaStreamSynchronize(ctx->stream);
            cudaStreamSynchronize(ctx->stream2);
            return KB_ERR_ARG;
        }
        const size_t m0 = (size_t)msg_off[lo], mb = (size_t)msg_off[hi] - m0;
        cudaStream_t st = pipe ? copy : lane[l];
        // lane l still holds chunk k-2: its kernels must have finished (its statuses were copied out behind the same event)
        if (pipe && k >= 2) KB_CUDA(cudaStreamWaitEvent(copy, ctx->pipe_done[l], 0));
        KB_CUDA(cudaMemcpyAsync(d_pk[l], pk + 32 * lo, 32 * cn, cudaMemcpyHostToDevice, st));
        KB_CUDA(cudaMemcpyAsync(d_sig[l], sig + 64 * lo, 64 * cn, cudaMemcpyHostToDevice, st));
        if (mb) KB_CUDA(cudaMemcpyAsync(d_m[l], msg + m0, mb, cudaMemcpyHostToDevice, st));
        KB_CUDA(cudaMemcpyAsync(d_off[l], msg_off + lo, 8 * (cn + 1), cudaMemcpyHostToDevice, st));
        if (pipe) {
            KB_CUDA(cudaEventRecord(ctx->pipe_ready[l], copy));
            KB_CUDA(cudaStreamWaitEvent(compute, ctx->pipe_ready[l], 0));
        }
        // offsets stay absolute; the kernel is told that d_m[l] starts at byte m0 of the caller's array
        int rc = kb_verify_launch(ctx, cn, d_pk[l], d_m[l], d_off[l], (uint64_t)m0, d_sig[l], d_st[l], schnorr, xyz[l], fl[l], pipe ? compute : st);
        if (rc != KB_OK) {
            cudaStreamSynchronize(ctx->stream);
            cudaStreamSynchronize(ctx->stream2);
            return rc;
        }
        if (pipe) {
            KB_CUDA(cudaEventRecord(ctx->pipe_done[l], compute));
            // the statuses of the PREVIOUS chunk leave behind this chunk's inputs: the copy stream never waits for kernels
            // that were enqueued after the copies it still has to do
            if (k >= 1) {
                KB_CUDA(cudaStreamWaitEvent(copy, ctx->pipe_done[l ^ 1], 0));
                KB_CUDA(cudaMemcpyAsync(status + cut[k - 1], d_st[l ^ 1], cut[k] - cut[k - 1], cudaMemcpyDeviceToHost, copy));
            }
        } else {
            KB_CUDA(cudaMemcpyAsync(status + lo, d_st[l], cn, cudaMemcpyDeviceToHost, st));
        }
    }
    if (pipe) {
        const int l = (int)((nchunks - 1) & 1);
        KB_CUDA(cudaStreamWaitEvent(copy, ctx->pipe_done[l], 0));
        KB_CUDA(cudaMemcpyAsync(status + cut[nchunks - 1], d_st[l], n - cut[nchunks - 1], cudaMemcpyDeviceToHost, copy));
    }
    KB_CUDA(cudaStreamSynchronize(ctx->stream));
    KB_CUDA(cudaStreamSynchronize(ctx->stream2));
    return KB_OK;
}
int kb_eddsa_verify_batch(kb_ctx* ctx, size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status)
{
    return kb_verify_host(ctx, n, pk, msg, msg_off, sig, status, 0);
}
int kb_schnorr_verify_batch(kb_ctx* ctx, size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status)
{
    return kb_verify_host(ctx, n, pk, msg, msg_off, sig, status, 1);
}

// device part of kb_eddsa_sign_batch; the caller wipes the secret scratch whatever this returns
static int kb_sign_run(kb_ctx* ctx, size_t n, const uint8_t* seeds, const uint8_t* msg, const uint64_t* msg_off, size_t mbytes, uint8_t* sig, uint8_t* pk, uint8_t* d_seed, uint8_t* d_a, uint8_t* d_r)
{
    uint8_t *d_m, *d_ra, *d_sig, *d_pk;
    uint64_t* d_off;
    uint32_t* xyz;
    KB_SCRATCH(4, mbytes, d_m);
    KB_SCRATCH(5, 8 * (n + 1), d_off);
    KB_SCRATCH(2, 64 * n, d_sig);
    KB_SCRATCH(1, 32 * n, d_pk);
    KB_SCRATCH(8, 64 * n, d_ra);
    KB_SCRATCH(KB_SLOT_XYZ, 96 * 2 * n, xyz);
    KB_H2D(d_seed, seeds, 32 * n);
    if (mbytes) KB_H2D(d_m, msg, mbytes);
    KB_H2D(d_off, msg_off, 8 * (n + 1));
    k_sign_stage1<<<kb_blocks(n, KB_THREADS), KB_THREADS, 64 * 8 * 96, ctx->stream>>>(n, d_seed, d_m, d_off, xyz, d_a, d_r, ctx->base_table);
    KB_LAUNCHED();
    k_compress_batch<<<kb_blocks((2 * n + KB_INV_K - 1) / KB_INV_K, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(2 * n, xyz, nullptr, d_ra);
    KB_LAUNCHED();
    k_sign_finish<<<kb_blocks(n, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(n, d_ra, d_m, d_off, d_a, d_r, d_sig, d_pk);
    KB_LAUNCHED();
    KB_D2H(sig, d_sig, 64 * n);
    if (pk) KB_D2H(pk, d_pk, 32 * n);
    return KB_OK;
}
int kb_eddsa_sign_batch(kb_ctx* ctx, size_t n, const uint8_t* seeds, const uint8_t* msg, const uint64_t* msg_off, uint8_t* sig, uint8_t* pk)
{
    KB_ENTER();
    if (n && (!seeds || !msg_off || !sig)) return KB_ERR_ARG;
    if (n == 0) return KB_OK;
    if (!kb_msg_off_ok(n, msg_off)) return KB_ERR_ARG;
    const size_t mbytes = (size_t)msg_off[n];
    if (mbytes && !msg) return KB_ERR_ARG;
    uint8_t *d_seed, *d_a, *d_r;
    KB_SCRATCH(0, 32 * n, d_seed);
    KB_SCRATCH(6, 32 * n, d_a);
    KB_SCRATCH(7, 32 * n, d_r);
    const int rc = kb_sign_run(ctx, n, seeds, msg, msg_off, mbytes, sig, pk, d_seed, d_a, d_r);
    // the secret scalars do not outlive the call, on the error paths either
    cudaMemsetAsync(d_a, 0, 32 * n, ctx->stream);
    cudaMemsetAsync(d_r, 0, 32 * n, ctx->stream);
    cudaMemsetAsync(d_seed, 0, 32 * n, ctx->stream);
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    KB_SYNC();
    return KB_OK;
}
int kb_verify_kernel_times(kb_ctx* ctx, int enable, float* ms_out)
{
    KB_ENTER();
    if (ms_out) {
        if (!ctx->timing || !ctx->timing_valid) return KB_ERR_ARG;
        KB_CUDA(cudaEventSynchronize(ctx->tev[2]));
        KB_CUDA(cudaEventElapsedTime(&ms_out[0], ctx->tev[0], ctx->tev[1]));
        KB_CUDA(cudaEventElapsedTime(&ms_out[1], ctx->tev[1], ctx->tev[2]));
    }
    ctx->timing = enable ? 1 : 0;
    if (!enable) ctx->timing_valid = 0;
    return KB_OK;
}

}  // extern "C"
