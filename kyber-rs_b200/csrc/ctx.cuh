// ctx.cuh — what the translation units of libkyber_b200.so share: the context, its growable device
// scratch and the error / launch bookkeeping macros.  Internal; the public contract is include/kyber_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/kyber_b200.h"
#include "ge.cuh"

#define KB_NSLOTS 64
#define KB_SLOT_XYZ 28
#define KB_SLOT_FLAGS 29

struct kb_ctx {
    int device;
    int sm_count;
    cudaStream_t stream;
    cudaStream_t stream2;    // second copy/compute lane of the pipelined host entry points
    ge_precomp* base_table;  // 64 x 8 entries: (j+1) * 16^w * B
    ge_precomp* base128;     // 128 entries: (j+1) * B (built only for the full-length verifiers, KB_VERIFY_FULL=1)
    ge_precomp* comb;        // KB_COMB_POS x KB_COMB_HALF entries: (j+1) * 2^(17 p) * B (94 MB)
    int verify_full;         // KB_VERIFY_FULL=1 in the environment: the full-length (253-doubling) verify kernels
    size_t verify_chunk;     // signatures per pipelined chunk of the host-buffer verify calls (KB_VERIFY_CHUNK_LOG2 overrides)
    int msm_c;               // KB_MSM_C: Pippenger window bits override (0 = by size)
    int msm_groups;          // KB_MSM_GROUPS: bucket groups per window in the Pippenger reduction (0 = default)
    int dkg_fd;              // KB_DKG_FD: 1 = always / 0 = never use the forward-difference DKG round (default: by cost)
    size_t fd_q4_max;        // KB_FD_Q4_MAX: conversion launches of up to this many cells run on four lanes per cell (default 8192)
    size_t fd_check_q4_max;  // KB_FD_CHECK_Q4_MAX: the same for the items of the final check (default 8192)
    int fd_graph;            // KB_FD_GRAPH: 1 (default) = the conversion chain is launched as a CUDA graph
    int fd_steps_wide, fd_steps_minb;   // KB_FD_STEPS_WIDE / KB_FD_STEPS_MINB: variants of the step kernel (tuning)
    int fd_parts;            // KB_FD_PARTS: number of coefficient blocks of the forward-difference round (0 = by cost)
    int verify_min_windows;  // KB_VERIFY_MIN_WINDOWS (tests): lower bound on the block-uniform window count of k_verify_half_main
    // KB_VERIFY_SPLIT: the preparation of the half-size-scalar verifiers as TWO kernels that share the SMs (capi_verify.cu):
    // a persistent ALU-bound "scalars" kernel (vs_blocks blocks per SM) beside the multiplier-bound "points" kernel
    int verify_split, vs_blocks, vs_pbound;
    cudaStream_t vs_side[2];                   // side stream per launch stream (the two lanes of the host-buffer pipeline)
    cudaEvent_t vs_fork[2], vs_join[2];
    unsigned long long* vs_counter;            // work counters of the persistent kernel, one per side stream
    int verify_sort;         // KB_VERIFY_SORT (default 1): the main kernel walks the records in the order of their loop lengths
    int verify_pipe;         // KB_VERIFY_PIPE: 0 = two independent lanes (default); 1 = kernels of all chunks on ONE stream, copies on the other
    size_t verify_chunk_n;   // KB_VERIFY_CHUNK: signatures per chunk as a plain count (overrides KB_VERIFY_CHUNK_LOG2)
    cudaEvent_t fork_ev, join_ev;              // a device entry point that runs two independent kernels side by side (Pippenger merge)
    cudaEvent_t pipe_ready[2], pipe_done[2];   // per staging lane: inputs copied in / kernels finished
    int timing;              // kb_verify_kernel_times: record events around the two launches of a device verify
    int timing_valid;
    cudaEvent_t tev[3];
    // Device entry points (kb_dev_*) of ONE context share its scratch slots.  Calls enqueued on different streams are
    // ordered through this event: every call first makes its stream wait for the previous call's end.
    cudaEvent_t order_ev;
    int order_valid;
    // x^(q h) mod 8L table of the forward-difference round (dkgfd.cuh), cached per (n, h, parts)
    uint32_t* fd_pw_host;    // pinned
    size_t fd_pw_host_words;
    size_t fd_pw_key[3];
    cudaEvent_t fd_pw_ev;    // end of the last upload from fd_pw_host
    // the chain of conversion launches of the forward-difference round as an instantiated CUDA graph, per shape (capi_poly.cu)
    void* fd_graph_exec;     // cudaGraphExec_t
    size_t fd_graph_nodes;
    size_t fd_graph_key[8];
    void* slot[KB_NSLOTS];
    size_t slot_bytes[KB_NSLOTS];
    uint64_t launches;
    char err[256];
};

static inline int kb_fail(kb_ctx* ctx, cudaError_t e, const char* what)
{
    if (ctx) snprintf(ctx->err, sizeof(ctx->err), "%s: %s", what, cudaGetErrorString(e));
    (void)cudaGetLastError();   // do not let this error be reported again by the next launch check
    return KB_ERR_CUDA;
}
#define KB_CUDA(call)                                              \
    do {                                                           \
        cudaError_t e_ = (call);                                   \
        if (e_ != cudaSuccess) return kb_fail(ctx, e_, #call);     \
    } while (0)
#define KB_LAUNCHED()                                              \
    do {                                                           \
        ctx->launches++;                                           \
        cudaError_t e_ = cudaGetLastError();                       \
        if (e_ != cudaSuccess) return kb_fail(ctx, e_, "launch");  \
    } while (0)

static inline unsigned kb_blocks(size_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }
// Block size of the long per-item kernels: a batch that fills the GPU less than about twice (config 1 is
// 2^16 items = 512 blocks of 128 on 148 SMs) is cut into 64-thread blocks so that the SMs end up evenly loaded.
static inline unsigned kb_item_threads(const kb_ctx* ctx, size_t n) { return n < (size_t)ctx->sm_count * 1024 ? 64u : 128u; }

// message offsets of a host-buffer call: msg_off[0..n] must be non-decreasing (message i is msg[msg_off[i] .. msg_off[i+1]));
// a kernel that met hi < lo would read out of bounds
static inline bool kb_msg_off_ok(size_t n, const uint64_t* msg_off)
{
    uint64_t bad = 0;
    for (size_t i = 0; i < n; i++) bad |= (uint64_t)(msg_off[i + 1] < msg_off[i]);
    return bad == 0;
}

// Growable device scratch buffer.  A slot only ever grows; growing frees and reallocates (which synchronises the
// device) — that happens on the first call of a given size, never in steady state.
int kb_scratch(kb_ctx* ctx, int s, size_t bytes, void** out);
#define KB_SCRATCH(s, bytes, ptr)                                          \
    do {                                                                   \
        void* p_;                                                          \
        int rc_ = kb_scratch(ctx, (s), (bytes), &p_);                      \
        if (rc_ != KB_OK) return rc_;                                      \
        (ptr) = reinterpret_cast<decltype(ptr)>(p_);                       \
    } while (0)

// host entry points: bind the device first
#define KB_ENTER()                                  \
    if (!ctx) return KB_ERR_ARG;                    \
    KB_CUDA(cudaSetDevice(ctx->device))
// device entry points: bind the device and order this call after the previous one of the context (shared scratch)
int kb_dev_begin(kb_ctx* ctx, cudaStream_t st);
int kb_dev_end(kb_ctx* ctx, cudaStream_t st);
#define KB_DEV_ENTER(st)                            \
    do {                                            \
        int rc_ = kb_dev_begin(ctx, (st));          \
        if (rc_ != KB_OK) return rc_;               \
    } while (0)
#define KB_DEV_RETURN(st, rc)                       \
    do {                                            \
        int rc2_ = (rc);                            \
        int rc3_ = kb_dev_end(ctx, (st));           \
        return rc2_ != KB_OK ? rc2_ : rc3_;         \
    } while (0)

#define KB_H2D(dst, src, bytes) KB_CUDA(cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyHostToDevice, ctx->stream))
#define KB_D2H(dst, src, bytes) KB_CUDA(cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyDeviceToHost, ctx->stream))
#define KB_SYNC() KB_CUDA(cudaStreamSynchronize(ctx->stream))

// Scratch slot map (one owner per slot within a call chain):
//   0..7    host-entry staging (inputs / outputs of kb_* calls)
//   8, 9    committed polynomials in cached form + bad flags (kb_poly_run); forward-difference array A / dealer flags
//   10..26, 53  Pippenger (msm);  27: multiplier table of the forward-difference round (cached across calls)
//   28, 29  KB_SLOT_XYZ / KB_SLOT_FLAGS: per-item intermediate points / flags
//   30, 31  forward-difference arrays B / decoded commitments
//   32..45  two lanes of the pipelined host-buffer verify
//   46..63  protocol-level entry points (capi_proto.cu) and the multi-device context

// ---- drivers shared between translation units (each defined in the file named) -------------------------------------
// capi_verify.cu: the two launches of a signature-verification batch on device buffers
int kb_verify_launch(kb_ctx* ctx, size_t n, const uint8_t* d_pk, const uint8_t* d_msg, const uint64_t* d_msg_off, uint64_t msg_base, const uint8_t* d_sig, uint8_t* d_status, int schnorr,
                     uint32_t* xyz, uint8_t* fl, cudaStream_t st);
// bytes per signature of the `xyz` scratch: one record of the half-size-scalar path (kernels.cuh), more than the 96 of the
// full-length path
#define KB_VERIFY_SCRATCH_BYTES (4 * KB_HALF_REC_WORDS)
// bytes of the `fl` scratch of kb_verify_launch: one flag byte per signature (full-length path) or, for the half-size-scalar
// path, the order in which the main kernel walks the records — uint32 perm[n], uint8 keys[n], 2 x 129 counters
#define KB_VERIFY_FLAG_BYTES(n) (5 * (size_t)(n) + 4096)
// capi_msm.cu: Pippenger on device buffers
// (ext != 0: the points are already decoded, 128 bytes each as X, Y, Z, T words)
int kb_msm_run(kb_ctx* ctx, size_t n, const uint8_t* d_scalars, const void* d_points, int ext, uint8_t* d_out32, uint32_t* d_partial128, unsigned long long* d_bad, cudaStream_t st);
// capi_poly.cu: a deal-verification round on device buffers (commitments as 32-byte encodings, or as the reference's
// 40-limb in-memory form when limbs != 0)
int kb_poly_run(kb_ctx* ctx, size_t npoly, size_t t, const void* d_commits, int limbs, size_t m, const uint32_t* d_poly_id, const uint32_t* d_idx, size_t n_verifiers,
                const uint8_t* d_shares, uint8_t* d_out, uint8_t* d_status, const uint32_t** d_xyz, cudaStream_t st);
int kb_dkg_round_run(kb_ctx* ctx, size_t n, size_t t, size_t ndealers, const void* d_commits, int limbs, const uint8_t* d_shares, uint8_t* d_verdict, cudaStream_t st);
