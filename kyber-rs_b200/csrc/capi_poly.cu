// capi_poly.cu — committed polynomials: PubPoly::eval / check, DKG deal-verification rounds, dkg_key
#define KB_K_POLY
#include "ctx.cuh"
#include "kernels.cuh"
#include "msm.cuh"
#include "dkgfd.cuh"
#include "dkgrlc.cuh"
#include "dkgcol.cuh"
#include <random>
// commitments -> cached form into scratch slots 8 (cached) / 9 (bad flags); then the eval kernel.
//   d_shares != 0           verdicts of the share checks into d_out (one byte per item)
//   d_shares == 0, d_out    encodings of the evaluations into d_out, per-item status into d_status
//   d_shares == 0, !d_out   the evaluations stay as (X, Y, Z) in scratch, *d_xyz points at them; status into d_status
int kb_poly_run(kb_ctx* ctx, size_t npoly, size_t t, const void* d_commits, int limbs, size_t m, const uint32_t* d_poly_id, const uint32_t* d_idx, size_t n_verifiers,
                       const uint8_t* d_shares, uint8_t* d_out, uint8_t* d_status, const uint32_t** d_xyz, cudaStream_t st)
{
    uint32_t* cached;
    uint8_t* bad;
    const size_t nc = npoly * t;
    KB_SCRATCH(8, nc * 128, cached);
    KB_SCRATCH(9, nc, bad);
    if (limbs) k_commit_prepare_limbs<<<kb_blocks(nc, KB_THREADS), KB_THREADS, 0, st>>>(nc, (const int32_t*)d_commits, cached, bad);
    else k_commit_prepare<<<kb_blocks(nc, KB_THREADS), KB_THREADS, 0, st>>>(nc, (const uint8_t*)d_commits, cached, bad);
    KB_LAUNCHED();
    if (d_shares) {
        k_poly_eval<<<kb_blocks(m, KB_THREADS), KB_THREADS, 64 * 8 * 96, st>>>(m, npoly, t, cached, bad, d_poly_id, d_idx, n_verifiers, d_shares, nullptr, nullptr, d_out, ctx->base_table);
        KB_LAUNCHED();
    } else {
        uint32_t* xyz;
        KB_SCRATCH(KB_SLOT_XYZ, 96 * m, xyz);
        k_poly_eval<<<kb_blocks(m, KB_THREADS), KB_THREADS, 0, st>>>(m, npoly, t, cached, bad, d_poly_id, d_idx, n_verifiers, nullptr, xyz, d_status, nullptr, ctx->base_table);
        KB_LAUNCHED();
        if (!d_out) {   // the caller goes on with the uncompressed values
            *d_xyz = xyz;
            return KB_OK;
        }
        k_compress_batch<<<kb_blocks((m + KB_INV_K - 1) / KB_INV_K, KB_THREADS), KB_THREADS, 0, st>>>(m, xyz, d_status, d_out);
        KB_LAUNCHED();
    }
    return KB_OK;
}
// The whole round by forward differences (dkgfd.cuh): one decode launch, h - 1 conversion launches, ONE launch for all
// n difference steps, one combine-and-check launch.
static int kb_dkg_fd_run(kb_ctx* ctx, size_t n, size_t t, size_t nd, size_t h, const void* d_commits, int limbs, const uint8_t* d_shares, uint8_t* d_verdict, cudaStream_t st)
{
    const size_t parts = (t + h - 1) / h;
    if (parts > KB_FD_MAX_PARTS || h > KB_FD_MAX_H) return KB_ERR_ARG;
    const size_t rows = parts * h;
    uint32_t *dec, *ra, *rb, *evals, *dbad, *pw;
    KB_SCRATCH(31, 128 * nd * t, dec);
    KB_SCRATCH(8, 128 * nd * rows, ra);
    KB_SCRATCH(30, 128 * nd * rows, rb);
    KB_SCRATCH(KB_SLOT_XYZ, 128 * parts * n * nd, evals);
    KB_SCRATCH(9, 4 * nd, dbad);
    const size_t pw_words = 9 * n * (parts - 1);
    KB_SCRATCH(27, 4 * pw_words, pw);
    if (parts > 1 && (ctx->fd_pw_key[0] != n || ctx->fd_pw_key[1] != h || ctx->fd_pw_key[2] != parts)) {
        // the public multipliers (i+1)^(q h) mod 8L: host integers, built when the shape of the round changes and kept
        // (in pinned memory and on the device) for the calls that follow
        KB_CUDA(cudaEventSynchronize(ctx->fd_pw_ev));   // an earlier upload may still be reading the pinned buffer
        if (ctx->fd_pw_host_words < pw_words) {
            if (ctx->fd_pw_host) cudaFreeHost(ctx->fd_pw_host);
            ctx->fd_pw_host = nullptr;
            ctx->fd_pw_host_words = 0;
            KB_CUDA(cudaMallocHost(&ctx->fd_pw_host, 4 * pw_words));
            ctx->fd_pw_host_words = pw_words;
        }
        kb_fd_power_table(n, h, parts, ctx->fd_pw_host);
        KB_CUDA(cudaMemcpyAsync(pw, ctx->fd_pw_host, 4 * pw_words, cudaMemcpyHostToDevice, st));
        KB_CUDA(cudaEventRecord(ctx->fd_pw_ev, st));
        ctx->fd_pw_key[0] = n;
        ctx->fd_pw_key[1] = h;
        ctx->fd_pw_key[2] = parts;
    }
    KB_CUDA(cudaMemsetAsync(dbad, 0, 4 * nd, st));
    if (limbs) k_fd_decode_limbs<<<kb_blocks(nd * t, KB_THREADS), KB_THREADS, 0, st>>>(nd, t, (const int32_t*)d_commits, dec, dbad);
    else k_fd_decode<<<kb_blocks(nd * t, KB_THREADS), KB_THREADS, 0, st>>>(nd, t, (const uint8_t*)d_commits, dec, dbad);
    KB_LAUNCHED();
    const size_t hl = kb_fd_part_len(t, h, parts - 1);
    const size_t q4_max = ctx->fd_q4_max;   // cells up to which a conversion launch uses four lanes per cell (KB_FD_Q4_MAX)
    // The h - 1 conversion launches form a chain in which every launch depends on the one before it and, for shards, lasts
    // a few microseconds: launched one by one they sit 2 - 2.7 us apart, as the nodes of a CUDA graph 0.5 us (measured on a
    // B200, tools/probe_graph.cu).  The chain only touches the context's scratch arrays, so it is built once per shape as an
    // explicit graph (kernel nodes in a line, no stream capture on the caller's stream) and kept with the context.
    const int use_graph = ctx->fd_graph;   // KB_FD_GRAPH
    const size_t gkey[8] = {nd, t, h, parts, q4_max, (size_t)dec, (size_t)ra, (size_t)rb};
    bool graph_ok = false;
    if (use_graph && h > 1) {
        if (!ctx->fd_graph_exec || memcmp(gkey, ctx->fd_graph_key, sizeof(gkey)) != 0) {
            if (ctx->fd_graph_exec) {
                cudaGraphExecDestroy((cudaGraphExec_t)ctx->fd_graph_exec);
                ctx->fd_graph_exec = nullptr;
            }
            cudaGraph_t g = nullptr;
            cudaGraphNode_t prev = nullptr;
            bool ok = cudaGraphCreate(&g, 0) == cudaSuccess;
            size_t nodes = 0;
            for (size_t s = 1; ok && s < h; s++) {
                const size_t sl = s + hl >= h ? s + hl - h : 0;
                const size_t cells = (parts - 1) * s + sl;
                if (cells == 0) continue;
                const uint32_t* src = (s & 1) ? rb : ra;
                uint32_t* dst = (s & 1) ? ra : rb;
                const bool q4 = q4_max && nd * cells <= q4_max;
                size_t a_nd = nd, a_t = t, a_h = h, a_parts = parts, a_s = s;
                const uint32_t* a_dec = dec;
                void* args[8] = {&a_nd, &a_t, &a_h, &a_parts, &a_s, &a_dec, &src, &dst};
                cudaKernelNodeParams kp;
                memset(&kp, 0, sizeof(kp));
                kp.func = q4 ? (void*)k_fd_conv_q4 : (void*)k_fd_conv;
                kp.gridDim = dim3(kb_blocks((q4 ? 4 : 1) * nd * cells, KB_FD_CONV_THREADS));
                kp.blockDim = dim3(KB_FD_CONV_THREADS);
                kp.kernelParams = args;
                cudaGraphNode_t node;
                ok = cudaGraphAddKernelNode(&node, g, prev ? &prev : nullptr, prev ? 1 : 0, &kp) == cudaSuccess;
                prev = node;
                nodes++;
            }
            cudaGraphExec_t ge = nullptr;
            ok = ok && nodes > 0 && cudaGraphInstantiate(&ge, g, 0) == cudaSuccess;
            if (g) cudaGraphDestroy(g);
            if (ok) {
                ctx->fd_graph_exec = ge;
                ctx->fd_graph_nodes = nodes;
                memcpy(ctx->fd_graph_key, gkey, sizeof(gkey));
            } else {
                (void)cudaGetLastError();   // fall through to the plain launches below
            }
        }
        if (ctx->fd_graph_exec && memcmp(gkey, ctx->fd_graph_key, sizeof(gkey)) == 0) {
            KB_CUDA(cudaGraphLaunch((cudaGraphExec_t)ctx->fd_graph_exec, st));
            ctx->launches += ctx->fd_graph_nodes;
            graph_ok = true;
        }
    }
    for (size_t s = 1; !graph_ok && s < h; s++) {
        const size_t sl = s + hl >= h ? s + hl - h : 0;
        const size_t cells = (parts - 1) * s + sl;
        if (cells == 0) continue;
        const uint32_t* src = (s & 1) ? rb : ra;
        uint32_t* dst = (s & 1) ? ra : rb;
        // few cells: the launch lasts one cell's latency — four lanes per cell shorten it (dkgfd.cuh).  Measured (round 2,
        // KB_FD_Q4_MAX sweep): the 32-dealer shard of config 3 (one rank of 8) 2.85 -> 2.33 ms with every launch on four lanes;
        // no gain from 128 dealers on, a loss when launches of more than ~10^4 cells use it (config 3 on one GPU: 5.9 -> 6.5 ms)
        if (q4_max && nd * cells <= q4_max) k_fd_conv_q4<<<kb_blocks(4 * nd * cells, KB_FD_CONV_THREADS), KB_FD_CONV_THREADS, 0, st>>>(nd, t, h, parts, s, dec, src, dst);
        else k_fd_conv<<<kb_blocks(nd * cells, KB_FD_CONV_THREADS), KB_FD_CONV_THREADS, 0, st>>>(nd, t, h, parts, s, dec, src, dst);
        KB_LAUNCHED();
    }
    const uint32_t* diffs = ((h - 1) & 1) ? ra : rb;   // what the last iteration wrote
    const unsigned step_threads = 32u * (unsigned)((h + 31) / 32);
    // up to 192 orders per block: 3 blocks (18 warps) per SM at 96 registers, or 4 at 80; up to 256: 2 blocks.
    // A whole round (thousands of blocks) runs equally fast with 2, 3 or 4 resident blocks per SM — the kernel is bound by the
    // multiplier pipe — but a SHARD's grid is a few blocks per SM and the launch lasts whole waves: 512 blocks (the 128 dealers
    // of one rank of 8) are 1.15 waves of 3 per SM and one wave of 4.  The variant whose waves cost less is launched.
    const int wide = ctx->fd_steps_wide;      // KB_FD_STEPS_WIDE: A/B switch (tuning)
    const int minb_env = ctx->fd_steps_minb;  // KB_FD_STEPS_MINB = 3 / 4: force a variant
    const size_t blocks = nd * parts, sms = (size_t)ctx->sm_count;
    const size_t waves3 = (blocks + 3 * sms - 1) / (3 * sms), waves4 = (blocks + 4 * sms - 1) / (4 * sms);
    const bool four = minb_env ? minb_env == 4 : (double)waves4 * 4.0 * 1.06 < (double)waves3 * 3.0;
    if (step_threads <= 192 && !wide) {
        if (four) k_fd_steps<192, 4><<<(unsigned)blocks, step_threads, 0, st>>>(nd, t, h, parts, n, dec, diffs, evals);
        else k_fd_steps<192, 3><<<(unsigned)blocks, step_threads, 0, st>>>(nd, t, h, parts, n, dec, diffs, evals);
    } else k_fd_steps<KB_FD_MAX_H, 2><<<(unsigned)blocks, step_threads, 0, st>>>(nd, t, h, parts, n, dec, diffs, evals);
    KB_LAUNCHED();
    // a few thousand items leave the GPU idle while each warp walks its ~450 dependent point operations: four lanes per item.
    // Measured (KB_FD_CHECK_Q4_MAX): a round of n = 64, t = 43 (4 096 items) 1.31 -> 1.08 ms; 8 192 items 2.24 -> 2.20 ms;
    // 16 384 items 2.32 -> 2.74 ms (slower: the table scans and conversions every lane repeats outweigh the shorter chain)
    const size_t cq4_max = ctx->fd_check_q4_max;   // KB_FD_CHECK_Q4_MAX
    if (nd * n <= cq4_max) k_fd_check_q4<<<kb_blocks(4 * nd * n, KB_THREADS), KB_THREADS, 64 * 8 * 96, st>>>(nd, n, parts, evals, pw, d_shares, dbad, ctx->base_table, d_verdict);
    else k_fd_check<<<kb_blocks(nd * n, KB_THREADS), KB_THREADS, 64 * 8 * 96, st>>>(nd, n, parts, evals, pw, d_shares, dbad, ctx->base_table, d_verdict);
    KB_LAUNCHED();
    return KB_OK;
}
// How to run a round: h = 0 means the per-share Horner kernel, otherwise forward differences with coefficient blocks of
// h.  Estimated from multiply counts (IMAD-eq) per dealer and the length of the chains of dependent launches / steps.
// The orders of a block are the lanes of k_fd_steps, so h is rounded up to whole warps where that keeps the block count.
static size_t kb_dkg_plan(const kb_ctx* ctx, size_t n, size_t t, size_t nd)
{
    if (ctx->dkg_fd == 0) return 0;
    const size_t pmin = (t + KB_FD_MAX_H - 1) / KB_FD_MAX_H;
    if (pmin > KB_FD_MAX_PARTS) return 0;
    const double rate = 7.0e12;   // sustained multiplies per second these kernels reach
    double best_time = 0;
    size_t best_h = 0, best_p = 0;
    for (size_t p = pmin ? pmin : 1; p <= KB_FD_MAX_PARTS && p <= t; p++) {
        if (ctx->fd_parts >= 1 && (size_t)ctx->fd_parts >= pmin && (size_t)ctx->fd_parts <= t && (size_t)ctx->fd_parts <= KB_FD_MAX_PARTS && p != (size_t)ctx->fd_parts) continue;
        size_t h = (t + p - 1) / p;
        const size_t h32 = (h + 31) / 32 * 32;
        if (h32 <= KB_FD_MAX_H && h32 < t && (t + h32 - 1) / h32 == (t + h - 1) / h) h = h32;
        const size_t pe = (t + h - 1) / h;
        double lg = 0;
        for (size_t x = h; x > 1; x >>= 1) lg += 1;
        const double cell = 900.0 + 590.0 * (lg > 1.5 ? lg - 1.5 : 0.0);
        double conv = 0, lanes = 0;
        for (size_t q = 0; q < pe; q++) {
            const double hq = (double)kb_fd_part_len(t, h, q);
            conv += 0.5 * hq * hq * cell;
            lanes += 32.0 * (double)((kb_fd_part_len(t, h, q) + 31) / 32);
        }
        const double steps = (double)n * lanes * 660.0 * 0.93;   // the dead orders of the last h steps are skipped
        const double comb = pe > 1 ? (double)n * (101000.0 + (pe - 1) * 42000.0) : 0.0;
        const double work = (conv + steps + comb + (double)n * 36000.0 + (double)t * 12700.0) * nd / rate;
        const double chain = h * 14e-6 + n * 2.5e-6 + (pe > 1 ? 0.3e-3 : 0.0);   // one cell per conversion launch, one addition per step, one Straus run
        const double time = work > chain ? work + 0.3 * chain : chain + 0.3 * work;
        if (best_h == 0 || time < best_time) {
            best_h = h;
            best_p = pe;
            best_time = time;
        }
    }
    if (best_h == 0) return 0;
    // its arrays: decoded commitments, two difference arrays, the recorded values — fall back to the per-share kernel
    // (a few MB of scratch) rather than fail when they would not fit next to what is already allocated
    {
        size_t free_b = 0, total_b = 0;
        const double need = 128.0 * nd * ((double)t + 2.0 * best_p * best_h + (double)best_p * n);
        const double have = (double)(ctx->slot_bytes[8] + ctx->slot_bytes[30] + ctx->slot_bytes[31] + ctx->slot_bytes[KB_SLOT_XYZ]);
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || need > 0.8 * (double)free_b + have) return 0;
    }
    if (ctx->dkg_fd == 1) return best_h;
    // the per-share kernel: one launch, but a thread walks all t coefficients (about 14 us each) on its own
    const double horner_work = ((double)n * t * 6800.0 + (double)n * 36000.0 + (double)t * 12700.0) * nd / rate;
    const double horner_chain = t * 14e-6 + 0.2e-3;
    const double horner = horner_work > horner_chain ? horner_work + 0.3 * horner_chain : horner_chain + 0.3 * horner_work;
    // measured, n = 256, t = 171: 32 / 64 / 128 / 256 dealers -> Horner 4.2 ms at 32 dealers, forward differences 2.5 / 3.5 / 5.8 ms
    return (nd * t >= 1024 && best_time * 1.15 < horner) ? best_h : 0;
}
// KB_ROUND_CHECK_BATCHED (dkgrlc.cuh): weights, decode, the shared-scalar multi-scalar multiplication, the torsion images and
// the share sums, one launch per dealer to decide, then the share-by-share checks of the dealers that failed, on a list
// whose length stays on the device.  Everything is enqueued on st; the fallback count is copied to rc_host at the end.
static int kb_dkg_rc_run(kb_ctx* ctx, size_t n, size_t t, size_t nd, const void* d_commits, int limbs, const uint8_t* d_shares, uint8_t* d_verdict, cudaStream_t st)
{
    ctx->rc_valid = 0;   // until this call has enqueued the copy of its own count
    if (nd >= ((size_t)1 << 32)) return KB_ERR_ARG;
    const size_t nd32 = (nd + 31) & ~(size_t)31, n32 = (n + 31) & ~(size_t)31;
    const size_t sms = (size_t)(ctx->sm_count > 0 ? ctx->sm_count : 1);
    // chunks per window: about 512 dealer-chunks per window, at most 2.  Measured on a B200 at 1 000 W (KB_RC_CHUNKS sweep of
    // tools/bench_round_batched.py, honest cfg4 round): 1 024 dealers 6.23 / 6.31 / 6.35 / 6.64 / 6.97 / 6.81 ms at 1 / 2 / 4 /
    // 5 / 8 / 16 chunks; the 128 dealers of one GPU of eight 3.19 / 2.47 / 2.64 / 2.89 / 3.21 / 3.80 ms.  More chunks fill the
    // GPU better in k_rc_msm but lengthen the fold in k_rc_dealer, a serial chain of one thread per dealer.
    size_t nch = ctx->rc_chunks ? (size_t)ctx->rc_chunks : (512 + nd32 - 1) / nd32;   // KB_RC_CHUNKS: 1..16
    if (!ctx->rc_chunks && nch > 2) nch = 2;
    if (nch > t) nch = t;
    if (nch < 1) nch = 1;
    // share sums: parts per dealer so that about four threads per SM-lane run, at most 32 and at most n
    size_t sparts = (4 * sms * 128 + nd - 1) / nd;
    if (sparts > 32) sparts = 32;
    if (sparts > n) sparts = n;
    if (sparts < 1) sparts = 1;
    uint32_t *dec, *dbad, *z, *ent, *cnt, *parts, *tor, *spart, *sflag, *stw, *list;
    unsigned long long* wacc;
    int16_t* dig;
    uint8_t* bkt;
    KB_SCRATCH(31, 128 * nd * t, dec);
    KB_SCRATCH(9, 4 * nd, dbad);
    KB_SCRATCH(55, 64 * t, wacc);
    KB_SCRATCH(56, 16 * n32, z);
    KB_SCRATCH(57, 2 * KB_RC_WINDOWS * t, dig);
    KB_SCRATCH(58, 4 * KB_RC_WINDOWS * t, ent);
    KB_SCRATCH(59, KB_RC_WINDOWS * t, bkt);
    KB_SCRATCH(60, 4 * (KB_RC_WINDOWS + 1 + 3 * nd), cnt);   // window counts, fallback count, state words, fallback list
    KB_SCRATCH(61, 128 * KB_RC_WINDOWS * nch * nd, parts);
    KB_SCRATCH(62, 128 * 5 * nd, tor);
    KB_SCRATCH(63, (32 + 4) * sparts * nd, spart);
    sflag = spart + 8 * sparts * nd;
    stw = cnt + KB_RC_WINDOWS + 1;
    list = stw + nd;
    // the weights are drawn after the inputs are in place, from the OS, for this call only
    kb_rc_seed seed;
    {
        std::random_device rd;
        for (int k = 0; k < 8; k++) seed.w[k] = (uint32_t)rd();
    }
    KB_CUDA(cudaMemsetAsync(wacc, 0, 64 * t, st));
    KB_CUDA(cudaMemsetAsync(dbad, 0, 4 * nd, st));
    const size_t jchunks = (t + KB_RC_POW_J - 1) / KB_RC_POW_J;
    k_rc_weights<<<kb_blocks(jchunks * n32, KB_THREADS), KB_THREADS, 0, st>>>(n, t, seed, z, wacc);
    KB_LAUNCHED();
    memset(&seed, 0, sizeof(seed));
    k_rc_digits<<<kb_blocks(t, KB_THREADS), KB_THREADS, 0, st>>>(t, wacc, dig);
    KB_LAUNCHED();
    k_rc_sort<<<KB_RC_WINDOWS, 256, 0, st>>>(t, dig, ent, bkt, cnt);
    KB_LAUNCHED();
    if (limbs) k_fd_decode_limbs<<<kb_blocks(nd * t, KB_THREADS), KB_THREADS, 0, st>>>(nd, t, (const int32_t*)d_commits, dec, dbad);
    else k_fd_decode<<<kb_blocks(nd * t, KB_THREADS), KB_THREADS, 0, st>>>(nd, t, (const uint8_t*)d_commits, dec, dbad);
    KB_LAUNCHED();
    // k_rc_torsion is a few blocks of long serial chains (t / 2 additions, then [L]): it runs on a second stream beside the
    // multi-scalar multiplication and the share sums, which fill the GPU
    cudaStream_t side = (st == ctx->stream2) ? ctx->stream : ctx->stream2;
    KB_CUDA(cudaEventRecord(ctx->fork_ev, st));
    KB_CUDA(cudaStreamWaitEvent(side, ctx->fork_ev, 0));
    k_rc_torsion<<<kb_blocks(5 * nd, KB_THREADS), KB_THREADS, 0, side>>>(nd, t, dec, tor);
    KB_LAUNCHED();
    KB_CUDA(cudaEventRecord(ctx->join_ev, side));
    k_rc_msm<<<kb_blocks(KB_RC_WINDOWS * nch * nd32, KB_THREADS), KB_THREADS, 0, st>>>(nd, t, nch, dec, ent, bkt, cnt, parts);
    KB_LAUNCHED();
    k_rc_shares<<<kb_blocks(sparts * nd, KB_THREADS), KB_THREADS, 0, st>>>(nd, n, sparts, z, d_shares, spart, sflag);
    KB_LAUNCHED();
    KB_CUDA(cudaStreamWaitEvent(st, ctx->join_ev, 0));
    k_rc_dealer<<<kb_blocks(nd, KB_THREADS), KB_THREADS, 64 * 8 * 96, st>>>(nd, nch, sparts, parts, tor, spart, sflag, dbad, ctx->base_table, stw);
    KB_LAUNCHED();
    // the sums of z_i s_(d,i) are combinations of the verifiers' secrets: they do not stay in device scratch
    KB_CUDA(cudaMemsetAsync(spart, 0, 32 * sparts * nd, st));
    k_rc_verdict<<<kb_blocks(nd * n, KB_THREADS), KB_THREADS, 0, st>>>(nd, n, stw, d_verdict);
    KB_LAUNCHED();
    k_rc_compact<<<1, 1024, 0, st>>>(nd, stw, list, cnt + KB_RC_WINDOWS);
    KB_LAUNCHED();
    k_poly_eval_list<<<kb_blocks(nd * n, KB_THREADS), KB_THREADS, 64 * 8 * 96, st>>>(nd, t, dec, dbad, list, cnt + KB_RC_WINDOWS, n, d_shares, d_verdict, ctx->base_table);
    KB_LAUNCHED();
    KB_CUDA(cudaMemcpyAsync(ctx->rc_host, cnt + KB_RC_WINDOWS, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    KB_CUDA(cudaEventRecord(ctx->rc_ev, st));
    ctx->rc_valid = 1;
    return KB_OK;
}
int kb_dkg_round_run(kb_ctx* ctx, size_t n, size_t t, size_t ndealers, const void* d_commits, int limbs, const uint8_t* d_shares, uint8_t* d_verdict, cudaStream_t st)
{
    if (ctx->round_check == KB_ROUND_CHECK_BATCHED) return kb_dkg_rc_run(ctx, n, t, ndealers, d_commits, limbs, d_shares, d_verdict, st);
    ctx->rc_valid = 0;
    const size_t h = kb_dkg_plan(ctx, n, t, ndealers);
    if (h) return kb_dkg_fd_run(ctx, n, t, ndealers, h, d_commits, limbs, d_shares, d_verdict, st);
    return kb_poly_run(ctx, ndealers, t, d_commits, limbs, n * ndealers, nullptr, nullptr, n, d_shares, d_verdict, nullptr, nullptr, st);
}
// (column, dealer) pairs per pass of the column kernel: its window sums take 128 * KB_COL_WINDOWS * chunks bytes per pair
// (138 MB per pass at one chunk), and 2^15 pairs are 33 windows x 2^15 threads, several times what the GPU holds
#define KB_COL_PAIRS ((size_t)1 << 15)
// How a partial verifier range is checked: the column kernel or the per-share Horner kernel on its items.  The column
// kernel costs about the same per (column, dealer) pair at any size, and 2.6 times a Horner walk once the GPU is full; the
// per-share kernel is bound by the latency of its walks (t dependent steps) until it has several items per lane.  Measured on
// a B200 at 1 000 W (tools/bench_dkg_columns.py, 1 024 dealers, t = 683, from ver_lo = 333): k = 1 / 4 / 6 / 8 / 16 / 64
// columns 4.9 / 12.8 / 18.5 / 22.5 / 42.9 / 166.0 ms by the column kernel, 15.4 / 17.4 / 19.3 / 19.4 / 24.0 / 82.8 ms per
// share; the two meet between 6 and 8 columns.  That was at x < 2^10: a Horner step is about one doubling per bit of x, so for larger x the crossover lies higher.
#define KB_COL_MAX_PAIRS ((size_t)6144)
static bool kb_dkg_columns_plan(const kb_ctx* ctx, size_t nd, size_t kc)
{
    if (ctx->dkg_columns >= 0) return ctx->dkg_columns != 0;   // KB_DKG_COLUMNS
    return nd * kc <= KB_COL_MAX_PAIRS;
}
// The share checks of verifiers [ver_lo, ver_hi) for nd dealers: shares and verdicts [d][kc], kc = ver_hi - ver_lo.  The
// whole range is the round itself.  A partial one runs the column kernel (dkgcol.cuh): one shared-exponent multi-scalar
// multiplication per column, in passes of at most KB_COL_PAIRS (column, dealer) pairs; or k_poly_eval on its items.
static int kb_dkg_columns_run(kb_ctx* ctx, size_t n, size_t t, size_t nd, size_t ver_lo, size_t ver_hi, const void* d_commits, int limbs, const uint8_t* d_shares, uint8_t* d_verdict,
                              cudaStream_t st)
{
    if (ver_lo == 0 && ver_hi == n) return kb_dkg_round_run(ctx, n, t, nd, d_commits, limbs, d_shares, d_verdict, st);
    ctx->rc_valid = 0;   // no share is checked twice: the fallback count of this call is 0
    const size_t kc = ver_hi - ver_lo;
    if (!kb_dkg_columns_plan(ctx, nd, kc)) {
        const size_t m = nd * kc;
        uint32_t *pid, *idx;
        KB_SCRATCH(55, 4 * m, pid);
        KB_SCRATCH(56, 4 * m, idx);
        k_col_items<<<kb_blocks(m, KB_THREADS), KB_THREADS, 0, st>>>(m, kc, ver_lo, pid, idx);
        KB_LAUNCHED();
        return kb_poly_run(ctx, nd, t, d_commits, limbs, m, pid, idx, 0, d_shares, d_verdict, nullptr, nullptr, st);
    }
    const size_t nd32 = (nd + 31) & ~(size_t)31;
    size_t group = KB_COL_PAIRS / nd;
    if (group < 1) group = 1;
    if (group > kc) group = kc;
    // chunks per window as kb_dkg_rc_run chooses them, counting the lanes of all the pass's columns
    size_t nch = ctx->rc_chunks ? (size_t)ctx->rc_chunks : (512 + group * nd32 - 1) / (group * nd32);   // KB_RC_CHUNKS: 1..16
    if (!ctx->rc_chunks && nch > 2) nch = 2;
    if (nch > t) nch = t;
    if (nch < 1) nch = 1;
    const size_t nwin = group * KB_COL_WINDOWS;
    uint32_t *dec, *dbad, *ent, *cnt, *parts;
    int16_t* dig;
    uint8_t* bkt;
    KB_SCRATCH(31, 128 * nd * t, dec);
    KB_SCRATCH(9, 4 * nd, dbad);
    KB_SCRATCH(57, 2 * nwin * t, dig);
    KB_SCRATCH(58, 4 * nwin * t, ent);
    KB_SCRATCH(59, nwin * t, bkt);
    KB_SCRATCH(60, 4 * nwin, cnt);
    KB_SCRATCH(61, 128 * nwin * nch * nd, parts);
    KB_CUDA(cudaMemsetAsync(dbad, 0, 4 * nd, st));
    if (limbs) k_fd_decode_limbs<<<kb_blocks(nd * t, KB_THREADS), KB_THREADS, 0, st>>>(nd, t, (const int32_t*)d_commits, dec, dbad);
    else k_fd_decode<<<kb_blocks(nd * t, KB_THREADS), KB_THREADS, 0, st>>>(nd, t, (const uint8_t*)d_commits, dec, dbad);
    KB_LAUNCHED();
    const size_t jchunks = (t + KB_RC_POW_J - 1) / KB_RC_POW_J;
    for (size_t c0 = 0; c0 < kc; c0 += group) {
        const size_t g = kc - c0 < group ? kc - c0 : group;
        k_col_digits<<<kb_blocks(g * jchunks, KB_THREADS), KB_THREADS, 0, st>>>(g, t, (uint64_t)(ver_lo + c0) + 1, dig);
        KB_LAUNCHED();
        k_rc_sort<<<(unsigned)(g * KB_COL_WINDOWS), 256, 0, st>>>(t, dig, ent, bkt, cnt);
        KB_LAUNCHED();
        k_col_msm<<<kb_blocks(g * KB_COL_WINDOWS * nch * nd32, KB_THREADS), KB_THREADS, 0, st>>>(nd, t, g * KB_COL_WINDOWS, nch, dec, ent, bkt, cnt, parts);
        KB_LAUNCHED();
        k_col_check<<<kb_blocks(g * nd, KB_THREADS), KB_THREADS, 64 * 8 * 96, st>>>(nd, g, kc, c0, nch, parts, dbad, d_shares, ctx->base_table, d_verdict);
        KB_LAUNCHED();
    }
    return KB_OK;
}
static bool kb_columns_args_ok(size_t n, size_t t, size_t nd_lo, size_t nd_hi, size_t ver_lo, size_t ver_hi, int fmt)
{
    return t && nd_lo <= nd_hi && ver_lo < ver_hi && ver_hi <= n && n <= ((size_t)1 << 32) && nd_hi - nd_lo < ((size_t)1 << 32) && t < ((size_t)1 << 31) &&
           (fmt == KB_POINT_ENC32 || fmt == KB_POINT_LIMBS40);
}

extern "C" {
int kb_dev_dkg_verify_round(kb_ctx* ctx, size_t n, size_t t, size_t ndealers, const void* d_commits, const void* d_shares, void* d_verdict, void* stream)
{
    if (!ctx || !t || (n && ndealers && (!d_commits || !d_shares || !d_verdict))) return KB_ERR_ARG;
    if (n == 0 || ndealers == 0) return KB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    KB_DEV_RETURN(st, kb_dkg_round_run(ctx, n, t, ndealers, d_commits, 0, (const uint8_t*)d_shares, (uint8_t*)d_verdict, st));
}
int kb_dev_dkg_verify_round_limbs(kb_ctx* ctx, size_t n, size_t t, size_t ndealers, const void* d_commit_limbs, const void* d_shares, void* d_verdict, void* stream)
{
    if (!ctx || !t || (n && ndealers && (!d_commit_limbs || !d_shares || !d_verdict))) return KB_ERR_ARG;
    if (n == 0 || ndealers == 0) return KB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    KB_DEV_RETURN(st, kb_dkg_round_run(ctx, n, t, ndealers, d_commit_limbs, 1, (const uint8_t*)d_shares, (uint8_t*)d_verdict, st));
}
static int kb_poly_host(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* commits, size_t m, const uint32_t* poly_id, const uint32_t* idx, const uint8_t* shares, uint8_t* out,
                        uint8_t* status)
{
    KB_ENTER();
    if (!npoly || !t || !commits || (m && (!poly_id || !idx || !out))) return KB_ERR_ARG;
    if (m == 0) return KB_OK;
    for (size_t k = 0; k < m; k++)
        if (poly_id[k] >= npoly) return KB_ERR_ARG;
    uint8_t *d_c, *d_sh = nullptr, *d_o, *d_st;
    uint32_t *d_pid, *d_idx;
    const size_t out_bytes = shares ? m : 32 * m;
    KB_SCRATCH(0, 32 * npoly * t, d_c);
    KB_SCRATCH(5, 4 * m, d_pid);
    KB_SCRATCH(6, 4 * m, d_idx);
    KB_SCRATCH(1, out_bytes, d_o);
    KB_SCRATCH(3, m, d_st);
    KB_H2D(d_c, commits, 32 * npoly * t);
    KB_H2D(d_pid, poly_id, 4 * m);
    KB_H2D(d_idx, idx, 4 * m);
    if (shares) {
        KB_SCRATCH(2, 32 * m, d_sh);
        KB_H2D(d_sh, shares, 32 * m);
    }
    int rc = kb_poly_run(ctx, npoly, t, d_c, 0, m, d_pid, d_idx, 0, d_sh, d_o, d_st, nullptr, ctx->stream);
    if (rc != KB_OK) return rc;
    KB_D2H(out, d_o, out_bytes);
    if (status && !shares) KB_D2H(status, d_st, m);
    KB_SYNC();
    return KB_OK;
}
int kb_pubpoly_eval_batch(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* commits, size_t m, const uint32_t* poly_id, const uint32_t* idx, uint8_t* out, uint8_t* status)
{
    return kb_poly_host(ctx, npoly, t, commits, m, poly_id, idx, nullptr, out, status);
}
int kb_vss_verify_deals_batch(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* commits, size_t m, const uint32_t* poly_id, const uint32_t* idx, const uint8_t* shares, uint8_t* verdict)
{
    if (m && !shares) return KB_ERR_ARG;
    return kb_poly_host(ctx, npoly, t, commits, m, poly_id, idx, shares, verdict, nullptr);
}
static int kb_dkg_round_host(kb_ctx* ctx, size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, const void* commits, int limbs, const uint8_t* shares, uint8_t* verdict)
{
    KB_ENTER();
    if (!t || dealer_hi < dealer_lo || !commits || !shares || !verdict) return KB_ERR_ARG;
    const size_t nd = dealer_hi - dealer_lo;
    if (nd == 0 || n == 0) return KB_OK;
    const size_t cbytes = limbs ? 160 : 32;   // per commitment
    uint8_t *d_c, *d_sh, *d_v;
    KB_SCRATCH(0, cbytes * nd * t, d_c);
    KB_SCRATCH(2, 32 * nd * n, d_sh);
    KB_SCRATCH(1, nd * n, d_v);
    KB_H2D(d_c, (const uint8_t*)commits + cbytes * dealer_lo * t, cbytes * nd * t);
    KB_H2D(d_sh, shares + 32 * dealer_lo * n, 32 * nd * n);
    int rc = kb_dkg_round_run(ctx, n, t, nd, d_c, limbs, d_sh, d_v, ctx->stream);
    // the shares are secrets of the verifiers: they do not stay in device scratch
    cudaMemsetAsync(d_sh, 0, 32 * nd * n, ctx->stream);
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    KB_D2H(verdict + dealer_lo * n, d_v, nd * n);
    KB_SYNC();
    return KB_OK;
}
int kb_dkg_verify_round(kb_ctx* ctx, size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, const uint8_t* commits, const uint8_t* shares, uint8_t* verdict)
{
    return kb_dkg_round_host(ctx, n, t, dealer_lo, dealer_hi, commits, 0, shares, verdict);
}
int kb_dkg_verify_round_limbs(kb_ctx* ctx, size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, const int32_t* commit_limbs, const uint8_t* shares, uint8_t* verdict)
{
    return kb_dkg_round_host(ctx, n, t, dealer_lo, dealer_hi, commit_limbs, 1, shares, verdict);
}
int kb_dkg_verify_columns(kb_ctx* ctx, size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, size_t ver_lo, size_t ver_hi, int fmt, const void* commits, const uint8_t* shares,
                          uint8_t* verdict)
{
    KB_ENTER();
    if (!kb_columns_args_ok(n, t, dealer_lo, dealer_hi, ver_lo, ver_hi, fmt)) return KB_ERR_ARG;
    const size_t nd = dealer_hi - dealer_lo, kc = ver_hi - ver_lo;
    if (nd == 0) return KB_OK;
    if (!commits || !shares || !verdict) return KB_ERR_ARG;
    const int limbs = fmt == KB_POINT_LIMBS40;
    const size_t cbytes = limbs ? 160 : 32;   // per commitment
    uint8_t *d_c, *d_sh, *d_v;
    KB_SCRATCH(0, cbytes * nd * t, d_c);
    KB_SCRATCH(2, 32 * nd * kc, d_sh);
    KB_SCRATCH(1, nd * kc, d_v);
    KB_H2D(d_c, (const uint8_t*)commits + cbytes * dealer_lo * t, cbytes * nd * t);
    KB_H2D(d_sh, shares, 32 * nd * kc);
    int rc = kb_dkg_columns_run(ctx, n, t, nd, ver_lo, ver_hi, d_c, limbs, d_sh, d_v, ctx->stream);
    // the shares are secrets of the verifiers: they do not stay in device scratch
    cudaMemsetAsync(d_sh, 0, 32 * nd * kc, ctx->stream);
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    KB_D2H(verdict, d_v, nd * kc);
    KB_SYNC();
    return KB_OK;
}
int kb_dev_dkg_verify_columns(kb_ctx* ctx, size_t n, size_t t, size_t ndealers, size_t ver_lo, size_t ver_hi, int fmt, const void* d_commits, const void* d_shares, void* d_verdict,
                              void* stream)
{
    if (!ctx || !kb_columns_args_ok(n, t, 0, ndealers, ver_lo, ver_hi, fmt)) return KB_ERR_ARG;
    if (ndealers == 0) return KB_OK;
    if (!d_commits || !d_shares || !d_verdict) return KB_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    KB_DEV_RETURN(st, kb_dkg_columns_run(ctx, n, t, ndealers, ver_lo, ver_hi, d_commits, fmt == KB_POINT_LIMBS40, (const uint8_t*)d_shares, (uint8_t*)d_verdict, st));
}

int kb_dev_pripoly_eval(kb_ctx* ctx, size_t npoly, size_t t, const void* d_coeffs, size_t n, void* d_out, void* stream)
{
    if (!ctx || !t || (npoly && n && (!d_coeffs || !d_out))) return KB_ERR_ARG;
    if (npoly == 0 || n == 0) return KB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    k_pripoly_eval<<<kb_blocks(npoly * n, KB_THREADS), KB_THREADS, 0, st>>>(npoly, t, (const uint8_t*)d_coeffs, n, (uint8_t*)d_out);
    KB_LAUNCHED();
    KB_DEV_RETURN(st, KB_OK);
}
int kb_pripoly_eval_batch(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* coeffs, size_t n, uint8_t* out)
{
    KB_ENTER();
    if (!t || (npoly && n && (!coeffs || !out))) return KB_ERR_ARG;
    if (npoly == 0 || n == 0) return KB_OK;
    uint8_t *d_c, *d_o;
    KB_SCRATCH(0, 32 * npoly * t, d_c);
    KB_SCRATCH(1, 32 * npoly * n, d_o);
    KB_H2D(d_c, coeffs, 32 * npoly * t);
    int rc = kb_dev_pripoly_eval(ctx, npoly, t, d_c, n, d_o, ctx->stream);
    cudaMemsetAsync(d_c, 0, 32 * npoly * t, ctx->stream);   // the private coefficients do not stay in device scratch
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    KB_D2H(out, d_o, 32 * npoly * n);
    KB_CUDA(cudaMemsetAsync(d_o, 0, 32 * npoly * n, ctx->stream));
    KB_SYNC();
    return KB_OK;
}

int kb_pubpoly_sum(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* commits, uint8_t* out, uint8_t* status)
{
    KB_ENTER();
    if (!npoly || !t || !commits || !out) return KB_ERR_ARG;
    const size_t nc = npoly * t;
    uint8_t *d_c, *bad, *d_o, *d_st;
    uint32_t *cached, *xyz;
    KB_SCRATCH(0, 32 * nc, d_c);
    KB_SCRATCH(8, 128 * nc, cached);
    KB_SCRATCH(9, nc, bad);
    KB_SCRATCH(KB_SLOT_XYZ, 96 * t, xyz);
    KB_SCRATCH(3, t, d_st);
    KB_SCRATCH(1, 32 * t, d_o);
    KB_H2D(d_c, commits, 32 * nc);
    k_commit_prepare<<<kb_blocks(nc, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(nc, d_c, cached, bad);
    KB_LAUNCHED();
    k_poly_colsum<<<kb_blocks(32 * t, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(npoly, t, cached, bad, xyz, d_st);
    KB_LAUNCHED();
    k_compress_batch<<<kb_blocks((t + KB_INV_K - 1) / KB_INV_K, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(t, xyz, d_st, d_o);
    KB_LAUNCHED();
    KB_D2H(out, d_o, 32 * t);
    if (status) KB_D2H(status, d_st, t);
    KB_SYNC();
    return KB_OK;
}

}  // extern "C"
