// capi_proto.cu — protocol-level entry points: the group math of the reference's DKG / VSS / DSS verifiers as whole
// operations, composed on the device from the kernels of the hot path (proto.cuh).
#define KB_K_POINT
#include "ctx.cuh"
#include "kernels.cuh"
#include "proto.cuh"

// n points in the caller's format (32-byte encodings or 40-limb elements, already on the device) -> canonical
// encodings (what marshal_binary returns) + bad flags; xyz = 96 n bytes of scratch
static int kb_canon_points(kb_ctx* ctx, size_t n, int fmt, const void* d_in, uint8_t* d_enc, uint8_t* d_bad, uint32_t* xyz, cudaStream_t st)
{
    if (n == 0) return KB_OK;
    if (fmt == KB_POINT_LIMBS40) k_points_from_limbs<<<kb_blocks(n, KB_THREADS), KB_THREADS, 0, st>>>(n, (const int32_t*)d_in, xyz, d_bad);
    else k_points_decode_xyz<<<kb_blocks(n, KB_THREADS), KB_THREADS, 0, st>>>(n, (const uint8_t*)d_in, xyz, d_bad);
    KB_LAUNCHED();
    k_compress_batch<<<kb_blocks((n + KB_INV_K - 1) / KB_INV_K, KB_THREADS), KB_THREADS, 0, st>>>(n, xyz, d_bad, d_enc);
    KB_LAUNCHED();
    return KB_OK;
}
static inline size_t kb_point_bytes(int fmt) { return fmt == KB_POINT_LIMBS40 ? 160 : 32; }

extern "C" {

int kb_vss_session_ids(kb_ctx* ctx, size_t ndealers, size_t n, size_t t, int fmt, const void* dealers, const void* verifiers, const void* commits, uint8_t* out32, uint8_t* status)
{
    KB_ENTER();
    if ((fmt != KB_POINT_ENC32 && fmt != KB_POINT_LIMBS40) || !out32 || (ndealers && (!dealers || (n && !verifiers) || (t && !commits)))) return KB_ERR_ARG;
    if (ndealers == 0) return KB_OK;
    const size_t pb = kb_point_bytes(fmt), total = ndealers + n + ndealers * t;
    uint8_t *d_in, *d_enc, *d_bad, *d_out, *d_st;
    uint32_t* xyz;
    KB_SCRATCH(46, pb * total, d_in);
    KB_SCRATCH(47, 32 * total, d_enc);
    KB_SCRATCH(48, total, d_bad);
    KB_SCRATCH(49, 33 * ndealers, d_out);
    d_st = d_out + 32 * ndealers;
    KB_SCRATCH(KB_SLOT_XYZ, 96 * total, xyz);
    KB_H2D(d_in, dealers, pb * ndealers);
    if (n) KB_H2D(d_in + pb * ndealers, verifiers, pb * n);
    if (t) KB_H2D(d_in + pb * (ndealers + n), commits, pb * ndealers * t);
    int rc = kb_canon_points(ctx, total, fmt, d_in, d_enc, d_bad, xyz, ctx->stream);
    if (rc != KB_OK) return rc;
    k_session_ids<<<kb_blocks(ndealers, 32), 32, 0, ctx->stream>>>(ndealers, n, t, d_enc, d_enc + 32 * ndealers, d_enc + 32 * (ndealers + n), d_bad, d_out, d_st);
    KB_LAUNCHED();
    KB_D2H(out32, d_out, 32 * ndealers);
    if (status) KB_D2H(status, d_st, ndealers);
    KB_SYNC();
    return KB_OK;
}

int kb_find_pub_batch(kb_ctx* ctx, size_t nlist, const void* list, size_t m, const void* queries, int fmt, int32_t* index_out)
{
    KB_ENTER();
    if ((fmt != KB_POINT_ENC32 && fmt != KB_POINT_LIMBS40) || (m && (!queries || !index_out)) || (nlist && !list)) return KB_ERR_ARG;
    if (m == 0) return KB_OK;
    const size_t pb = kb_point_bytes(fmt), total = nlist + m;
    uint8_t *d_in, *d_enc, *d_bad;
    int32_t* d_idx;
    uint32_t* xyz;
    KB_SCRATCH(46, pb * total, d_in);
    KB_SCRATCH(47, 32 * total, d_enc);
    KB_SCRATCH(48, total, d_bad);
    KB_SCRATCH(49, 4 * m, d_idx);
    KB_SCRATCH(KB_SLOT_XYZ, 96 * total, xyz);
    if (nlist) KB_H2D(d_in, list, pb * nlist);
    KB_H2D(d_in + pb * nlist, queries, pb * m);
    int rc = kb_canon_points(ctx, total, fmt, d_in, d_enc, d_bad, xyz, ctx->stream);
    if (rc != KB_OK) return rc;
    k_find_pub<<<kb_blocks(m, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(nlist, d_enc, d_bad, m, d_enc + 32 * nlist, d_bad + nlist, d_idx);
    KB_LAUNCHED();
    KB_D2H(index_out, d_idx, 4 * m);
    KB_SYNC();
    return KB_OK;
}

// One DKG deal-verification round on device buffers: the n^2 share checks of the dealers given, then the Schnorr
// verification of their deal signatures and of the responses to them.  A signature batch with d_sig == 0 is skipped.
int kb_dev_dkg_process_round(kb_ctx* ctx, size_t n, size_t t, size_t ndealers, int fmt, const void* d_commits, const void* d_shares, void* d_verdict,
                             const void* d_deal_pk, const void* d_deal_msg, const void* d_deal_msg_off, const void* d_deal_sig, void* d_deal_status,
                             const void* d_resp_pk, const void* d_resp_msg, const void* d_resp_msg_off, const void* d_resp_sig, void* d_resp_status, void* stream)
{
    if (!ctx || !t || (fmt != KB_POINT_ENC32 && fmt != KB_POINT_LIMBS40) || (n && ndealers && (!d_commits || !d_shares || !d_verdict))) return KB_ERR_ARG;
    if (d_deal_sig && (!d_deal_pk || !d_deal_msg_off || !d_deal_status)) return KB_ERR_ARG;
    if (d_resp_sig && (!d_resp_pk || !d_resp_msg_off || !d_resp_status)) return KB_ERR_ARG;
    const size_t m = n * ndealers;
    if (m == 0) return KB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    KB_DEV_ENTER(st);
    int rc = kb_dkg_round_run(ctx, n, t, ndealers, d_commits, fmt == KB_POINT_LIMBS40, (const uint8_t*)d_shares, (uint8_t*)d_verdict, st);
    if (rc != KB_OK) return rc;
    uint32_t* xyz;
    uint8_t* fl;
    KB_SCRATCH(KB_SLOT_XYZ, (size_t)KB_VERIFY_SCRATCH_BYTES * m, xyz);
    KB_SCRATCH(KB_SLOT_FLAGS, KB_VERIFY_FLAG_BYTES(m), fl);
    if (d_deal_sig) {
        rc = kb_verify_launch(ctx, m, (const uint8_t*)d_deal_pk, (const uint8_t*)d_deal_msg, (const uint64_t*)d_deal_msg_off, 0, (const uint8_t*)d_deal_sig, (uint8_t*)d_deal_status, 1, xyz, fl, st);
        if (rc != KB_OK) return rc;
    }
    if (d_resp_sig) {
        rc = kb_verify_launch(ctx, m, (const uint8_t*)d_resp_pk, (const uint8_t*)d_resp_msg, (const uint64_t*)d_resp_msg_off, 0, (const uint8_t*)d_resp_sig, (uint8_t*)d_resp_status, 1, xyz, fl, st);
        if (rc != KB_OK) return rc;
    }
    KB_DEV_RETURN(st, KB_OK);
}
int kb_dkg_process_round(kb_ctx* ctx, size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, int fmt, const void* commits, const uint8_t* shares, uint8_t* verdict,
                         const uint8_t* deal_pk, const uint8_t* deal_msg, const uint64_t* deal_msg_off, const uint8_t* deal_sig, uint8_t* deal_status,
                         const uint8_t* resp_pk, const uint8_t* resp_msg, const uint64_t* resp_msg_off, const uint8_t* resp_sig, uint8_t* resp_status)
{
    if (!ctx || dealer_hi < dealer_lo) return KB_ERR_ARG;
    const size_t m = (dealer_hi - dealer_lo) * n;
    int rc;
    if (fmt == KB_POINT_LIMBS40) rc = kb_dkg_verify_round_limbs(ctx, n, t, dealer_lo, dealer_hi, (const int32_t*)commits, shares, verdict);
    else if (fmt == KB_POINT_ENC32) rc = kb_dkg_verify_round(ctx, n, t, dealer_lo, dealer_hi, (const uint8_t*)commits, shares, verdict);
    else return KB_ERR_ARG;
    if (rc != KB_OK) return rc;
    // the signature arrays hold the m = (dealer_hi - dealer_lo) * n items of this dealer range, item (d - dealer_lo) * n + i
    if (deal_sig) {
        rc = kb_schnorr_verify_batch(ctx, m, deal_pk, deal_msg, deal_msg_off, deal_sig, deal_status);
        if (rc != KB_OK) return rc;
    }
    if (resp_sig) rc = kb_schnorr_verify_batch(ctx, m, resp_pk, resp_msg, resp_msg_off, resp_sig, resp_status);
    return rc;
}

int kb_vss_rabin_verify_deals_batch(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* commits, const uint8_t* h_point, size_t m, const uint32_t* poly_id, const uint32_t* idx,
                                    const uint8_t* f_shares, const uint8_t* g_shares, uint8_t* verdict)
{
    KB_ENTER();
    if (!npoly || !t || !commits || !h_point || (m && (!poly_id || !idx || !f_shares || !g_shares || !verdict))) return KB_ERR_ARG;
    if (m == 0) return KB_OK;
    for (size_t k = 0; k < m; k++)
        if (poly_id[k] >= npoly) return KB_ERR_ARG;
    uint8_t *d_c, *d_f, *d_g, *d_h, *d_v, *d_st;
    uint32_t *d_pid, *d_idx;
    KB_SCRATCH(0, 32 * npoly * t, d_c);
    KB_SCRATCH(5, 4 * m, d_pid);
    KB_SCRATCH(6, 4 * m, d_idx);
    KB_SCRATCH(2, 32 * m, d_f);
    KB_SCRATCH(4, 32 * m, d_g);
    KB_SCRATCH(7, 32, d_h);
    KB_SCRATCH(1, m, d_v);
    KB_SCRATCH(3, m, d_st);
    KB_H2D(d_c, commits, 32 * npoly * t);
    KB_H2D(d_pid, poly_id, 4 * m);
    KB_H2D(d_idx, idx, 4 * m);
    KB_H2D(d_f, f_shares, 32 * m);
    KB_H2D(d_g, g_shares, 32 * m);
    KB_H2D(d_h, h_point, 32);
    const uint32_t* evals;
    int rc = kb_poly_run(ctx, npoly, t, d_c, 0, m, d_pid, d_idx, 0, nullptr, nullptr, d_st, &evals, ctx->stream);
    if (rc == KB_OK) {
        k_rabin_finish<<<kb_blocks(m, KB_THREADS), KB_THREADS, 64 * 8 * 96, ctx->stream>>>(m, evals, d_st, d_f, d_g, d_h, ctx->base_table, d_v);
        ctx->launches++;
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = kb_fail(ctx, e, "launch");
    }
    // the two shares are secrets of the verifier
    cudaMemsetAsync(d_f, 0, 32 * m, ctx->stream);
    cudaMemsetAsync(d_g, 0, 32 * m, ctx->stream);
    if (rc != KB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    KB_D2H(verdict, d_v, m);
    KB_SYNC();
    return KB_OK;
}

int kb_dss_verify_partials(kb_ctx* ctx, size_t t, const uint8_t* random_commits, const uint8_t* long_commits, const uint8_t* msg, size_t msg_len, size_t m, const uint32_t* idx, const uint8_t* partials,
                           uint8_t* verdict, uint8_t* hash_out32)
{
    KB_ENTER();
    if (!t || !random_commits || !long_commits || (msg_len && !msg) || (m && (!idx || !partials || !verdict))) return KB_ERR_ARG;
    uint8_t *d_c, *d_m, *d_ra, *d_rabad, *d_hash, *d_p, *d_v, *d_st;
    uint32_t *d_pid, *d_idx, *xyz2;
    uint64_t* d_off;
    KB_SCRATCH(0, 64 * t, d_c);
    KB_SCRATCH(4, msg_len, d_m);
    KB_SCRATCH(5, 4 * 2 * (m + 1), d_pid);
    KB_SCRATCH(6, 4 * 2 * (m + 1), d_idx);
    KB_SCRATCH(2, 32 * (m + 1), d_p);
    KB_SCRATCH(7, 64 + 2 + 32 + 16, d_ra);
    d_rabad = d_ra + 64;
    d_hash = d_ra + 80;                      // 16-byte aligned
    KB_SCRATCH(46, 16, d_off);
    KB_SCRATCH(47, 96 * 2, xyz2);
    KB_SCRATCH(1, m + 1, d_v);
    KB_SCRATCH(3, 2 * (m + 1), d_st);
    KB_H2D(d_c, random_commits, 32 * t);
    KB_H2D(d_c + 32 * t, long_commits, 32 * t);
    if (msg_len) KB_H2D(d_m, msg, msg_len);
    // hash = H(R || A || msg) with R, A the canonical encodings of the two free coefficients (hash_sig, dss_sig.rs:312-326)
    {
        const uint64_t off[2] = {0, (uint64_t)msg_len};
        KB_CUDA(cudaMemcpyAsync(d_off, off, 16, cudaMemcpyHostToDevice, ctx->stream));
        KB_CUDA(cudaStreamSynchronize(ctx->stream));   // `off` is on this stack frame
        KB_CUDA(cudaMemcpyAsync(d_ra, d_c, 32, cudaMemcpyDeviceToDevice, ctx->stream));
        KB_CUDA(cudaMemcpyAsync(d_ra + 32, d_c + 32 * t, 32, cudaMemcpyDeviceToDevice, ctx->stream));
        int rc = kb_canon_points(ctx, 2, KB_POINT_ENC32, d_ra, d_ra, d_rabad, xyz2, ctx->stream);
        if (rc != KB_OK) return rc;
        k_challenge<<<1, KB_THREADS, 0, ctx->stream>>>(1, d_ra, d_ra + 32, d_m, d_off, d_hash);
        KB_LAUNCHED();
        if (hash_out32) KB_D2H(hash_out32, d_hash, 32);
    }
    if (m) {
        // 2 m evaluations: items [0, m) the random polynomial (poly 0), [m, 2m) the long-term one (poly 1)
        uint32_t* hp = (uint32_t*)malloc(4 * 4 * m);
        if (!hp) return KB_ERR_NOMEM;
        for (size_t k = 0; k < m; k++) {
            hp[k] = 0;
            hp[m + k] = 1;
            hp[2 * m + k] = idx[k];
            hp[3 * m + k] = idx[k];
        }
        cudaError_t e = cudaMemcpyAsync(d_pid, hp, 8 * m, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_idx, hp + 2 * m, 8 * m, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        free(hp);
        if (e != cudaSuccess) return kb_fail(ctx, e, "dss index upload");
        KB_H2D(d_p, partials, 32 * m);
        const uint32_t* evals;
        int rc = kb_poly_run(ctx, 2, t, d_c, 0, 2 * m, d_pid, d_idx, 0, nullptr, nullptr, d_st, &evals, ctx->stream);
        if (rc != KB_OK) return rc;
        k_dss_finish<<<kb_blocks(m, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(m, evals, d_st, d_hash, d_p, ctx->comb, d_v);
        KB_LAUNCHED();
        KB_D2H(verdict, d_v, m);
    }
    KB_SYNC();
    return KB_OK;
}

// out[c] = sum_i lam_i * points[c][i] for the Lagrange coefficients lam of the nodes idx (device part shared by
// kb_recover_commit_batch and kb_dkg_resharing_key); d_points = ncols x k encodings, column-major as [c][i]
static int kb_recover_run(kb_ctx* ctx, size_t ncols, size_t k, const uint32_t* d_idx, const uint8_t* d_points, uint8_t* d_out, uint8_t* d_status, cudaStream_t st)
{
    uint8_t *d_lam, *d_bad;
    uint32_t *d_prod, *xyz;
    KB_SCRATCH(50, 32 * k, d_lam);
    KB_SCRATCH(51, 128 * ncols * k, d_prod);
    KB_SCRATCH(52, ncols * k, d_bad);
    KB_SCRATCH(KB_SLOT_XYZ, 96 * ncols, xyz);
    k_lagrange_coeffs<<<kb_blocks(k, KB_THREADS), KB_THREADS, 0, st>>>(k, d_idx, d_lam);
    KB_LAUNCHED();
    k_wmul<<<kb_blocks(ncols * k, KB_THREADS), KB_THREADS, 0, st>>>(ncols, k, d_lam, 0, d_points, 1, d_prod, d_bad);
    KB_LAUNCHED();
    k_colsum<<<kb_blocks(32 * ncols, KB_THREADS), KB_THREADS, 0, st>>>(ncols, k, d_prod, d_bad, xyz, d_status);
    KB_LAUNCHED();
    k_compress_batch<<<kb_blocks((ncols + KB_INV_K - 1) / KB_INV_K, KB_THREADS), KB_THREADS, 0, st>>>(ncols, xyz, d_status, d_out);
    KB_LAUNCHED();
    return KB_OK;
}
static bool kb_idx_distinct(size_t k, const uint32_t* idx)
{
    // the nodes of an interpolation must be distinct (a zero denominator otherwise); k is at most a few thousand
    for (size_t i = 0; i < k; i++)
        for (size_t j = i + 1; j < k; j++)
            if (idx[i] == idx[j]) return false;
    return true;
}

int kb_recover_commit_batch(kb_ctx* ctx, size_t ncols, size_t k, const uint32_t* idx, const uint8_t* points, uint8_t* out, uint8_t* status)
{
    KB_ENTER();
    if (!ncols || !k || !idx || !points || !out || !kb_idx_distinct(k, idx)) return KB_ERR_ARG;
    uint32_t* d_idx;
    uint8_t *d_pts, *d_o, *d_st;
    KB_SCRATCH(5, 4 * k, d_idx);
    KB_SCRATCH(0, 32 * ncols * k, d_pts);
    KB_SCRATCH(1, 32 * ncols, d_o);
    KB_SCRATCH(3, ncols, d_st);
    KB_H2D(d_idx, idx, 4 * k);
    KB_H2D(d_pts, points, 32 * ncols * k);
    int rc = kb_recover_run(ctx, ncols, k, d_idx, d_pts, d_o, d_st, ctx->stream);
    if (rc != KB_OK) return rc;
    KB_D2H(out, d_o, 32 * ncols);
    if (status) KB_D2H(status, d_st, ncols);
    KB_SYNC();
    return KB_OK;
}

int kb_recover_pub_poly(kb_ctx* ctx, size_t k, const uint32_t* idx, const uint8_t* points, uint8_t* out, uint8_t* status)
{
    KB_ENTER();
    if (!k || k > 1023 || !idx || !points || !out || !kb_idx_distinct(k, idx)) return KB_ERR_ARG;
    uint32_t *d_idx, *d_prod, *xyz;
    uint8_t *d_pts, *d_o, *d_st, *d_basis, *d_bad;
    KB_SCRATCH(5, 4 * k, d_idx);
    KB_SCRATCH(0, 32 * k, d_pts);
    KB_SCRATCH(1, 32 * k, d_o);
    KB_SCRATCH(3, k, d_st);
    KB_SCRATCH(50, 32 * k * k, d_basis);
    KB_SCRATCH(51, 128 * k * k, d_prod);
    KB_SCRATCH(52, k * k, d_bad);
    KB_SCRATCH(KB_SLOT_XYZ, 96 * k, xyz);
    KB_H2D(d_idx, idx, 4 * k);
    KB_H2D(d_pts, points, 32 * k);
    k_lagrange_basis<<<1, (unsigned)(k + 1), 32 * (k + 1), ctx->stream>>>(k, d_idx, d_basis);
    KB_LAUNCHED();
    // coefficient c of the result = sum_j basis_j[c] * y_j  (basis.commit(y_j) added up, poly.rs:620-632)
    k_wmul<<<kb_blocks(k * k, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(k, k, d_basis, 1, d_pts, 0, d_prod, d_bad);
    KB_LAUNCHED();
    k_colsum<<<kb_blocks(32 * k, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(k, k, d_prod, d_bad, xyz, d_st);
    KB_LAUNCHED();
    k_compress_batch<<<kb_blocks((k + KB_INV_K - 1) / KB_INV_K, KB_THREADS), KB_THREADS, 0, ctx->stream>>>(k, xyz, d_st, d_o);
    KB_LAUNCHED();
    KB_D2H(out, d_o, 32 * k);
    if (status) KB_D2H(status, d_st, k);
    KB_SYNC();
    return KB_OK;
}

int kb_dkg_resharing_key(kb_ctx* ctx, size_t new_t, size_t k, const uint32_t* idx, const uint8_t* coeffs, uint32_t share_idx, const uint8_t* share32, uint8_t* out_commits, uint8_t* status, uint8_t* check_out)
{
    KB_ENTER();
    if (!new_t || !k || !idx || !coeffs || !out_commits || !kb_idx_distinct(k, idx)) return KB_ERR_ARG;
    uint32_t *d_idx, *d_one;
    uint8_t *d_in, *d_pts, *d_o, *d_st, *d_sh, *d_v;
    KB_SCRATCH(5, 4 * k + 16, d_idx);
    KB_SCRATCH(46, 32 * new_t * k, d_in);
    KB_SCRATCH(0, 32 * new_t * k, d_pts);
    KB_SCRATCH(1, 32 * new_t, d_o);
    KB_SCRATCH(3, new_t, d_st);
    KB_SCRATCH(2, 32, d_sh);
    KB_SCRATCH(6, 16, d_one);
    KB_SCRATCH(7, 16, d_v);
    KB_H2D(d_idx, idx, 4 * k);
    KB_H2D(d_in, coeffs, 32 * new_t * k);
    // coeffs[i][c] (the deal of qualified node i holds new_t commitments) -> points[c][i] (dkg.rs:1003-1016)
    k_transpose32<<<kb_blocks(new_t * k, 256), 256, 0, ctx->stream>>>(k, new_t, d_in, d_pts);
    KB_LAUNCHED();
    int rc = kb_recover_run(ctx, new_t, k, d_idx, d_pts, d_o, d_st, ctx->stream);
    if (rc != KB_OK) return rc;
    KB_D2H(out_commits, d_o, 32 * new_t);
    if (status) KB_D2H(status, d_st, new_t);
    if (share32 && check_out) {
        // pub_poly.check(private_share) (dkg.rs:1029-1031): one evaluation of the new polynomial against share * B
        const uint32_t hv[2] = {0u, share_idx};
        KB_CUDA(cudaMemcpyAsync(d_one, hv, 8, cudaMemcpyHostToDevice, ctx->stream));
        KB_H2D(d_sh, share32, 32);
        KB_CUDA(cudaStreamSynchronize(ctx->stream));   // hv is on this stack frame
        rc = kb_poly_run(ctx, 1, new_t, d_o, 0, 1, d_one, d_one + 1, 0, d_sh, d_v, nullptr, nullptr, ctx->stream);
        cudaMemsetAsync(d_sh, 0, 32, ctx->stream);
        if (rc != KB_OK) {
            cudaStreamSynchronize(ctx->stream);
            return rc;
        }
        KB_D2H(check_out, d_v, 1);
    }
    KB_SYNC();
    return KB_OK;
}

}  // extern "C"
