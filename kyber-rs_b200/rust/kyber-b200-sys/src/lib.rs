//! `extern "C"` declarations for `include/kyber_b200.h` — one per exported symbol.
//! NOT COMPILED in the environment this repository is built in (no rustc/cargo); kept in
//! lock-step with the header by `tests/test_abi_cpu.py::test_rust_sys_matches_header`.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_double, c_int, c_void};

#[repr(C)]
pub struct kb_ctx {
    _private: [u8; 0],
}

#[repr(C)]
pub struct kb_keyset {
    _private: [u8; 0],
}

#[repr(C)]
pub struct kb_mctx {
    _private: [u8; 0],
}

#[repr(C)]
pub struct kb_mkeyset {
    _private: [u8; 0],
}

#[repr(C)]
pub struct kb_signerset {
    _private: [u8; 0],
}

#[repr(C)]
pub struct kb_msignerset {
    _private: [u8; 0],
}

pub const KB_SIGNER_SCHNORR: c_int = 0;
pub const KB_SIGNER_EDDSA: c_int = 1;

pub const KB_OK: c_int = 0;
pub const KB_ERR_NCCL: c_int = -4;
pub const KB_ERR_ARG: c_int = -1;
pub const KB_ERR_CUDA: c_int = -2;
pub const KB_ERR_NOMEM: c_int = -3;
pub const KB_FLAG_VARTIME: u32 = 1;
pub const KB_FLAG_SHARED_POINT: u32 = 2;

#[link(name = "kyber_b200")]
extern "C" {
    pub fn kb_ctx_create(device: c_int, out: *mut *mut kb_ctx) -> c_int;
    pub fn kb_ctx_destroy(ctx: *mut kb_ctx);
    pub fn kb_ctx_wipe(ctx: *mut kb_ctx) -> c_int;
    pub fn kb_last_error(ctx: *const kb_ctx) -> *const c_char;
    pub fn kb_device_sm_count(ctx: *const kb_ctx) -> c_int;
    pub fn kb_launch_count(ctx: *const kb_ctx) -> u64;
    pub fn kb_host_alloc(bytes: usize) -> *mut c_void;
    pub fn kb_host_free(p: *mut c_void);

    pub fn kb_point_mul_base_batch(ctx: *mut kb_ctx, n: usize, scalars: *const u8, out: *mut u8, flags: u32) -> c_int;
    pub fn kb_point_mul_batch(ctx: *mut kb_ctx, n: usize, scalars: *const u8, points: *const u8, out: *mut u8, status: *mut u8, flags: u32) -> c_int;
    pub fn kb_point_recode_batch(ctx: *mut kb_ctx, n: usize, input: *const u8, out: *mut u8, status: *mut u8) -> c_int;
    pub fn kb_point_from_limbs_batch(ctx: *mut kb_ctx, n: usize, limbs: *const i32, out: *mut u8) -> c_int;
    pub fn kb_point_add_batch(ctx: *mut kb_ctx, n: usize, p: *const u8, q: *const u8, out: *mut u8, status: *mut u8, subtract: c_int) -> c_int;
    pub fn kb_point_check_batch(ctx: *mut kb_ctx, n: usize, input: *const u8, flags_out: *mut u8) -> c_int;
    pub fn kb_point_decompress_batch(ctx: *mut kb_ctx, n: usize, input: *const u8, out128: *mut u8, status: *mut u8) -> c_int;
    pub fn kb_point_compress_batch(ctx: *mut kb_ctx, n: usize, in128: *const u8, out: *mut u8) -> c_int;
    pub fn kb_point_eq_batch(ctx: *mut kb_ctx, n: usize, p: *const u8, q: *const u8, equal_out: *mut u8) -> c_int;

    pub fn kb_sc_reduce64_batch(ctx: *mut kb_ctx, n: usize, in64: *const u8, out32: *mut u8) -> c_int;
    pub fn kb_sc_muladd_batch(ctx: *mut kb_ctx, n: usize, a: *const u8, b: *const u8, c: *const u8, out: *mut u8) -> c_int;
    pub fn kb_sc_invert_batch(ctx: *mut kb_ctx, n: usize, a: *const u8, out: *mut u8) -> c_int;
    pub fn kb_challenge_batch(ctx: *mut kb_ctx, n: usize, r32: *const u8, a32: *const u8, msg: *const u8, msg_off: *const u64, out32: *mut u8) -> c_int;

    pub fn kb_eddsa_verify_batch(ctx: *mut kb_ctx, n: usize, pk: *const u8, msg: *const u8, msg_off: *const u64, sig: *const u8, status: *mut u8) -> c_int;
    pub fn kb_schnorr_verify_batch(ctx: *mut kb_ctx, n: usize, pk: *const u8, msg: *const u8, msg_off: *const u64, sig: *const u8, status: *mut u8) -> c_int;

    // key sets: verification under registered public keys
    pub fn kb_keyset_create(ctx: *mut kb_ctx, nkeys: usize, pk: *const u8, out: *mut *mut kb_keyset) -> c_int;
    pub fn kb_keyset_destroy(ks: *mut kb_keyset);
    pub fn kb_keyset_verify_batch(ks: *mut kb_keyset, n: usize, key_idx: *const u32, msg: *const u8, msg_off: *const u64, sig: *const u8, status: *mut u8, schnorr: c_int) -> c_int;
    pub fn kb_dev_keyset_verify(ks: *mut kb_keyset, n: usize, d_key_idx: *const c_void, d_msg: *const c_void, d_msg_off: *const c_void, d_sig: *const c_void, d_status: *mut c_void, schnorr: c_int, stream: *mut c_void) -> c_int;
    pub fn kb_keyset_verify_pk_batch(ks: *mut kb_keyset, n: usize, pk: *const u8, msg: *const u8, msg_off: *const u64, sig: *const u8, status: *mut u8, schnorr: c_int, hits: *mut u64) -> c_int;
    pub fn kb_dev_keyset_verify_pk(ks: *mut kb_keyset, n: usize, d_pk: *const c_void, d_msg: *const c_void, d_msg_off: *const c_void, d_sig: *const c_void, d_status: *mut c_void, schnorr: c_int, d_hits: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn kb_keyset_mul_batch(ks: *mut kb_keyset, n: usize, key_idx: *const u32, scalars: *const u8, out: *mut u8, status: *mut u8, flags: u32) -> c_int;
    pub fn kb_dev_keyset_mul(ks: *mut kb_keyset, n: usize, d_key_idx: *const c_void, d_scalars: *const c_void, d_out: *mut c_void, d_status: *mut c_void, flags: u32, stream: *mut c_void) -> c_int;

    pub fn kb_eddsa_sign_batch(ctx: *mut kb_ctx, n: usize, seeds: *const u8, msg: *const u8, msg_off: *const u64, sig: *mut u8, pk: *mut u8) -> c_int;
    pub fn kb_schnorr_sign_batch(ctx: *mut kb_ctx, n: usize, secrets: *const u8, nonces: *const u8, msg: *const u8, msg_off: *const u64, sig: *mut u8, pk: *mut u8) -> c_int;
    pub fn kb_dev_schnorr_sign(ctx: *mut kb_ctx, n: usize, d_secrets: *const c_void, d_nonces: *const c_void, d_msg: *const c_void, d_msg_off: *const c_void, d_sig: *mut c_void, d_pk: *mut c_void, stream: *mut c_void) -> c_int;
    // signer sets: signing under registered secret keys (kind: KB_SIGNER_SCHNORR or KB_SIGNER_EDDSA)
    pub fn kb_signerset_create(ctx: *mut kb_ctx, nkeys: usize, keys: *const u8, kind: c_int, pk_out: *mut u8, out: *mut *mut kb_signerset) -> c_int;
    pub fn kb_signerset_destroy(ss: *mut kb_signerset);
    pub fn kb_signerset_sign_batch(ss: *mut kb_signerset, n: usize, key_idx: *const u32, nonces: *const u8, msg: *const u8, msg_off: *const u64, sig: *mut u8) -> c_int;
    pub fn kb_dev_signerset_sign(ss: *mut kb_signerset, n: usize, d_key_idx: *const c_void, d_nonces: *const c_void, d_msg: *const c_void, d_msg_off: *const c_void, d_sig: *mut c_void, d_status: *mut c_void, stream: *mut c_void) -> c_int;

    pub fn kb_pubpoly_eval_batch(ctx: *mut kb_ctx, npoly: usize, t: usize, commits: *const u8, m: usize, poly_id: *const u32, idx: *const u32, out: *mut u8, status: *mut u8) -> c_int;
    pub fn kb_vss_verify_deals_batch(ctx: *mut kb_ctx, npoly: usize, t: usize, commits: *const u8, m: usize, poly_id: *const u32, idx: *const u32, shares: *const u8, verdict: *mut u8) -> c_int;
    pub fn kb_dkg_verify_round(ctx: *mut kb_ctx, n: usize, t: usize, dealer_lo: usize, dealer_hi: usize, commits: *const u8, shares: *const u8, verdict: *mut u8) -> c_int;
    pub fn kb_dkg_verify_round_limbs(ctx: *mut kb_ctx, n: usize, t: usize, dealer_lo: usize, dealer_hi: usize, commit_limbs: *const i32, shares: *const u8, verdict: *mut u8) -> c_int;
    pub fn kb_dkg_verify_columns(ctx: *mut kb_ctx, n: usize, t: usize, dealer_lo: usize, dealer_hi: usize, ver_lo: usize, ver_hi: usize, fmt: c_int, commits: *const c_void, shares: *const u8, verdict: *mut u8) -> c_int;
    pub fn kb_ctx_set_round_check(ctx: *mut kb_ctx, mode: c_int) -> c_int;
    pub fn kb_ctx_round_fallbacks(ctx: *mut kb_ctx, dealers: *mut u64) -> c_int;

    pub fn kb_pubpoly_sum(ctx: *mut kb_ctx, npoly: usize, t: usize, commits: *const u8, out: *mut u8, status: *mut u8) -> c_int;

    pub fn kb_msm(ctx: *mut kb_ctx, n: usize, scalars: *const u8, points: *const u8, out32: *mut u8, partial128: *mut u8, bad_points: *mut u64) -> c_int;
    pub fn kb_point_sum(ctx: *mut kb_ctx, k: usize, partials128: *const u8, out32: *mut u8) -> c_int;

    // protocol-level operations (fmt: 0 = 32-byte encodings, 1 = 40 x i32 limbs per point)
    pub fn kb_vss_session_ids(ctx: *mut kb_ctx, ndealers: usize, n: usize, t: usize, fmt: c_int, dealers: *const c_void, verifiers: *const c_void, commits: *const c_void, out32: *mut u8, status: *mut u8) -> c_int;
    pub fn kb_find_pub_batch(ctx: *mut kb_ctx, nlist: usize, list: *const c_void, m: usize, queries: *const c_void, fmt: c_int, index_out: *mut i32) -> c_int;
    pub fn kb_dkg_process_round(ctx: *mut kb_ctx, n: usize, t: usize, dealer_lo: usize, dealer_hi: usize, fmt: c_int, commits: *const c_void, shares: *const u8, verdict: *mut u8,
        deal_pk: *const u8, deal_msg: *const u8, deal_msg_off: *const u64, deal_sig: *const u8, deal_status: *mut u8,
        resp_pk: *const u8, resp_msg: *const u8, resp_msg_off: *const u64, resp_sig: *const u8, resp_status: *mut u8) -> c_int;
    pub fn kb_vss_rabin_verify_deals_batch(ctx: *mut kb_ctx, npoly: usize, t: usize, commits: *const u8, h_point: *const u8, m: usize, poly_id: *const u32, idx: *const u32, f_shares: *const u8, g_shares: *const u8, verdict: *mut u8) -> c_int;
    pub fn kb_dss_verify_partials(ctx: *mut kb_ctx, t: usize, random_commits: *const u8, long_commits: *const u8, msg: *const u8, msg_len: usize, m: usize, idx: *const u32, partials: *const u8, verdict: *mut u8, hash_out32: *mut u8) -> c_int;
    pub fn kb_recover_commit_batch(ctx: *mut kb_ctx, ncols: usize, k: usize, idx: *const u32, points: *const u8, out: *mut u8, status: *mut u8) -> c_int;
    pub fn kb_recover_pub_poly(ctx: *mut kb_ctx, k: usize, idx: *const u32, points: *const u8, out: *mut u8, status: *mut u8) -> c_int;
    pub fn kb_dkg_resharing_key(ctx: *mut kb_ctx, new_t: usize, k: usize, idx: *const u32, coeffs: *const u8, share_idx: u32, share32: *const u8, out_commits: *mut u8, status: *mut u8, check_out: *mut u8) -> c_int;
    pub fn kb_dev_dkg_process_round(ctx: *mut kb_ctx, n: usize, t: usize, ndealers: usize, fmt: c_int, d_commits: *const c_void, d_shares: *const c_void, d_verdict: *mut c_void,
        d_deal_pk: *const c_void, d_deal_msg: *const c_void, d_deal_msg_off: *const c_void, d_deal_sig: *const c_void, d_deal_status: *mut c_void,
        d_resp_pk: *const c_void, d_resp_msg: *const c_void, d_resp_msg_off: *const c_void, d_resp_sig: *const c_void, d_resp_status: *mut c_void, stream: *mut c_void) -> c_int;
    // DKG rounds under registered participant keys (deal k: dealer key dealer_lo + k / n, response k: verifier key k % n)
    pub fn kb_dkg_process_round_keyed(ctx: *mut kb_ctx, dealers: *const kb_keyset, verifiers: *const kb_keyset, n: usize, t: usize, dealer_lo: usize, dealer_hi: usize, fmt: c_int,
        commits: *const c_void, shares: *const u8, verdict: *mut u8,
        deal_msg: *const u8, deal_msg_off: *const u64, deal_sig: *const u8, deal_status: *mut u8,
        resp_msg: *const u8, resp_msg_off: *const u64, resp_sig: *const u8, resp_status: *mut u8) -> c_int;
    pub fn kb_dev_dkg_process_round_keyed(ctx: *mut kb_ctx, dealers: *const kb_keyset, verifiers: *const kb_keyset, n: usize, t: usize, dealer_lo: usize, ndealers: usize, fmt: c_int,
        d_commits: *const c_void, d_shares: *const c_void, d_verdict: *mut c_void,
        d_deal_msg: *const c_void, d_deal_msg_off: *const c_void, d_deal_sig: *const c_void, d_deal_status: *mut c_void,
        d_resp_msg: *const c_void, d_resp_msg_off: *const c_void, d_resp_sig: *const c_void, d_resp_status: *mut c_void, stream: *mut c_void) -> c_int;

    pub fn kb_dev_eddsa_verify(ctx: *mut kb_ctx, n: usize, d_pk: *const c_void, d_msg: *const c_void, d_msg_off: *const c_void, d_sig: *const c_void, d_status: *mut c_void, schnorr: c_int, stream: *mut c_void) -> c_int;
    pub fn kb_dev_point_mul_base(ctx: *mut kb_ctx, n: usize, d_scalars: *const c_void, d_out: *mut c_void, flags: u32, stream: *mut c_void) -> c_int;
    pub fn kb_dev_point_mul(ctx: *mut kb_ctx, n: usize, d_scalars: *const c_void, d_points: *const c_void, d_out: *mut c_void, d_status: *mut c_void, flags: u32, stream: *mut c_void) -> c_int;
    pub fn kb_dev_msm(ctx: *mut kb_ctx, n: usize, d_scalars: *const c_void, d_points: *const c_void, d_out32: *mut c_void, d_partial128: *mut c_void, d_bad_points: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn kb_dev_msm_ext(ctx: *mut kb_ctx, n: usize, d_scalars: *const c_void, d_points128: *const c_void, d_out32: *mut c_void, d_partial128: *mut c_void, d_bad_points: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn kb_dev_dkg_verify_round(ctx: *mut kb_ctx, n: usize, t: usize, ndealers: usize, d_commits: *const c_void, d_shares: *const c_void, d_verdict: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn kb_dev_dkg_verify_round_limbs(ctx: *mut kb_ctx, n: usize, t: usize, ndealers: usize, d_commit_limbs: *const c_void, d_shares: *const c_void, d_verdict: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn kb_dev_dkg_verify_columns(ctx: *mut kb_ctx, n: usize, t: usize, ndealers: usize, ver_lo: usize, ver_hi: usize, fmt: c_int, d_commits: *const c_void, d_shares: *const c_void, d_verdict: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn kb_dev_point_sum(ctx: *mut kb_ctx, k: usize, d_partials128: *const c_void, d_out32: *mut c_void, stream: *mut c_void) -> c_int;

    pub fn kb_pripoly_eval_batch(ctx: *mut kb_ctx, npoly: usize, t: usize, coeffs: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn kb_dev_pripoly_eval(ctx: *mut kb_ctx, npoly: usize, t: usize, d_coeffs: *const c_void, n: usize, d_out: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn kb_dev_point_decompress(ctx: *mut kb_ctx, n: usize, d_in: *const c_void, d_out128: *mut c_void, d_status: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn kb_dev_challenge(ctx: *mut kb_ctx, n: usize, d_r32: *const c_void, d_a32: *const c_void, d_msg: *const c_void, d_msg_off: *const c_void, d_out32: *mut c_void, stream: *mut c_void) -> c_int;
    // multi-device context
    pub fn kb_mctx_create(devices: *const c_int, ndev: c_int, out: *mut *mut kb_mctx) -> c_int;
    pub fn kb_mctx_destroy(m: *mut kb_mctx);
    pub fn kb_mctx_device_count(m: *const kb_mctx) -> c_int;
    pub fn kb_mctx_ctx(m: *mut kb_mctx, i: c_int) -> *mut kb_ctx;
    pub fn kb_mctx_last_error(m: *const kb_mctx) -> *const c_char;
    pub fn kb_mctx_launch_count(m: *const kb_mctx) -> u64;
    pub fn kb_mctx_verify_batch(m: *mut kb_mctx, n: usize, pk: *const u8, msg: *const u8, msg_off: *const u64, sig: *const u8, status: *mut u8, schnorr: c_int) -> c_int;
    pub fn kb_mctx_point_mul_base_batch(m: *mut kb_mctx, n: usize, scalars: *const u8, out: *mut u8, flags: u32) -> c_int;
    pub fn kb_mctx_point_mul_batch(m: *mut kb_mctx, n: usize, scalars: *const u8, points: *const u8, out: *mut u8, status: *mut u8, flags: u32) -> c_int;
    pub fn kb_mctx_dkg_verify_round(m: *mut kb_mctx, n: usize, t: usize, ndealers: usize, fmt: c_int, commits: *const c_void, shares: *const u8, verdict: *mut u8) -> c_int;
    pub fn kb_mctx_dkg_process_round(m: *mut kb_mctx, n: usize, t: usize, ndealers: usize, fmt: c_int, commits: *const c_void, shares: *const u8, verdict: *mut u8,
        deal_pk: *const u8, deal_msg: *const u8, deal_msg_off: *const u64, deal_sig: *const u8, deal_status: *mut u8,
        resp_pk: *const u8, resp_msg: *const u8, resp_msg_off: *const u64, resp_sig: *const u8, resp_status: *mut u8) -> c_int;
    pub fn kb_mctx_keyset_create(m: *mut kb_mctx, nkeys: usize, pk: *const u8, out: *mut *mut kb_mkeyset) -> c_int;
    pub fn kb_mctx_keyset_destroy(ks: *mut kb_mkeyset);
    pub fn kb_mctx_keyset_verify_batch(ks: *mut kb_mkeyset, n: usize, key_idx: *const u32, msg: *const u8, msg_off: *const u64, sig: *const u8, status: *mut u8, schnorr: c_int) -> c_int;
    pub fn kb_mctx_keyset_verify_pk_batch(ks: *mut kb_mkeyset, n: usize, pk: *const u8, msg: *const u8, msg_off: *const u64, sig: *const u8, status: *mut u8, schnorr: c_int, hits: *mut u64) -> c_int;
    pub fn kb_mctx_keyset_mul_batch(ks: *mut kb_mkeyset, n: usize, key_idx: *const u32, scalars: *const u8, out: *mut u8, status: *mut u8, flags: u32) -> c_int;
    pub fn kb_mctx_dkg_process_round_keyed(m: *mut kb_mctx, dealers: *const kb_mkeyset, verifiers: *const kb_mkeyset, n: usize, t: usize, ndealers: usize, fmt: c_int,
        commits: *const c_void, shares: *const u8, verdict: *mut u8,
        deal_msg: *const u8, deal_msg_off: *const u64, deal_sig: *const u8, deal_status: *mut u8,
        resp_msg: *const u8, resp_msg_off: *const u64, resp_sig: *const u8, resp_status: *mut u8) -> c_int;
    pub fn kb_mctx_schnorr_sign_batch(m: *mut kb_mctx, n: usize, secrets: *const u8, nonces: *const u8, msg: *const u8, msg_off: *const u64, sig: *mut u8, pk: *mut u8) -> c_int;
    pub fn kb_mctx_signerset_create(m: *mut kb_mctx, nkeys: usize, keys: *const u8, kind: c_int, pk_out: *mut u8, out: *mut *mut kb_msignerset) -> c_int;
    pub fn kb_mctx_signerset_destroy(ss: *mut kb_msignerset);
    pub fn kb_mctx_signerset_sign_batch(ss: *mut kb_msignerset, n: usize, key_idx: *const u32, nonces: *const u8, msg: *const u8, msg_off: *const u64, sig: *mut u8) -> c_int;
    pub fn kb_mctx_msm(m: *mut kb_mctx, n: usize, scalars: *const u8, points: *const u8, out32: *mut u8, bad_points: *mut u64) -> c_int;

    pub fn kb_probe_imad(ctx: *mut kb_ctx, kind: c_int, iters: c_int, macs_per_sec: *mut c_double, elapsed_ms: *mut c_double) -> c_int;
    pub fn kb_verify_kernel_times(ctx: *mut kb_ctx, enable: c_int, ms_out: *mut f32) -> c_int;
}
