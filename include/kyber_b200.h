/*
 * kyber_b200.h — C ABI of the B200-native edwards25519 hot path of teleconsys/kyber-rs.
 *
 * This is the drop-in boundary (SURVEY §8b).  kyber-rs has no FFI of its own; the seam is
 * its generic trait surface (src/group.rs: Scalar :22, Point :85, Group :185) that every
 * protocol module is generic over.  A `kyber-b200-sys` crate binds exactly these symbols
 * (see INTEGRATION.md) and adds batch methods behind the same traits.  Each entry point
 * names the reference interface it replaces (paths relative to /root/reference/src).
 *
 * Conventions
 *  - Points and scalars cross the ABI in the reference's own wire encoding: 32-byte
 *    compressed points (Point::marshal_binary, group/edwards25519/point.rs:35-41) and
 *    32-byte little-endian scalars (Scalar.v, scalar.rs:24).  Scalars are used as raw
 *    integers, never reduced mod L on entry (SURVEY §A3), exactly like Point::mul.
 *  - All buffers are caller-owned.  `kb_*` functions take HOST pointers, copy in, run the
 *    CUDA kernels, copy out and return after the device has finished.  `kb_dev_*` functions
 *    take DEVICE pointers plus a CUDA stream (cudaStream_t as void*, NULL = default stream)
 *    and only enqueue work; nothing is retained after return.  They use the context's scratch
 *    buffers, which grow (cudaMalloc, a device synchronisation) the first time a larger batch is
 *    seen and never in steady state; calls of one context on DIFFERENT streams are ordered one
 *    after the other by the library (a shared event), so they are safe but do not overlap.
 *  - Return value: KB_OK or a negative kb_err.  Per-item outcomes go to status arrays.
 *  - There is no CPU fallback: with no usable CUDA device every call fails with
 *    KB_ERR_CUDA.
 *  - A context is bound to one CUDA device and is not thread-safe; use one per host thread
 *    (the reference is single-threaded, group.rs has no shared mutable state).
 */
#ifndef KYBER_B200_H
#define KYBER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Environment switches read once by kb_ctx_create (tests, tuning and A/B measurements; none changes a result):
 *   KB_VERIFY_FULL=1          signature verifiers: the full-length (253-doubling) kernels instead of the half-size-scalar ones
 *   KB_VERIFY_MIN_WINDOWS=k   half-size-scalar verifier: lower bound on the block-uniform window count (tests)
 *   KB_VERIFY_CHUNK=n         host-buffer verify calls: largest pipelined chunk in signatures (default: 16 waves of the main
 *                             kernel = 16 x SMs x 512; the chunks grow x4 from a third of a wave up to this cap)
 *   KB_VERIFY_CHUNK_LOG2=k    the same cap as a power of two
 *   KB_VERIFY_PIPE=1          host-buffer verify calls: kernels of all chunks on one stream and copies on a second one
 *                             (default 0: two alternating lanes, each copy in / kernels / copy out)
 *   KB_VERIFY_SORT=0|2        half-size-scalar verifier: never / always hand the records to the main kernel sorted by loop length
 *                             (default 1: batches of 16384 signatures or more)
 *   KB_VERIFY_SPLIT=1|2       half-size-scalar verifier: the preparation as two kernels side by side — a persistent "scalars"
 *                             kernel of KB_VERIFY_SPLIT_BLOCKS (1..8, default 1) blocks per SM on a side stream beside the "points"
 *                             grid — for batches of at least one block per SM (1) or every batch (2); default 0: one kernel with
 *                             both phases (faster, see DESIGN 3.6)
 *   KB_DKG_FD=0|1             kb_dkg_verify_round: never / always by forward differences (default: by cost)
 *   KB_FD_PARTS=p             forward-difference round: cut each polynomial into p coefficient blocks, 1..4 (default: by cost)
 *   KB_FD_GRAPH=0             forward-difference round: launch the conversion chain kernel by kernel instead of as a CUDA graph
 *   KB_FD_CHECK_Q4_MAX=c      forward-difference round: the final check uses four lanes per item up to c items (default 8192, 0 = never)
 *   KB_FD_Q4_MAX=c            forward-difference round: conversion launches of up to c cells use four lanes per cell (default 8192, 0 = never)
 *   KB_MSM_C=c                Pippenger window bits (default floor(log2 n) - 3 within 4..16) */
typedef struct kb_ctx kb_ctx;

typedef enum kb_err {
    KB_OK = 0,
    KB_ERR_ARG = -1,   /* null pointer / bad size / bad flag */
    KB_ERR_CUDA = -2,  /* CUDA runtime error; kb_last_error() has the text */
    KB_ERR_NOMEM = -3,
    KB_ERR_NCCL = -4   /* NCCL could not be loaded or failed (multi-device context only) */
} kb_err;

/* Per-signature outcome; mirrors SignatureError (sign/error.rs:6-25) in the order the
 * respective verifier reports it. */
typedef enum kb_sig_status {
    KB_SIG_STATUS_OK = 0,
    KB_SIG_STATUS_LENGTH = 1,            /* InvalidSignatureLength (host-side mirror only) */
    KB_SIG_STATUS_NOT_CANONICAL = 2,     /* SignatureNotCanonical  */
    KB_SIG_STATUS_R_NOT_CANONICAL = 3,   /* RNotCanonical          */
    KB_SIG_STATUS_R_SMALL_ORDER = 4,     /* RSmallOrder            */
    KB_SIG_STATUS_PK_NOT_CANONICAL = 5,  /* PublicKeyNotCanonical  */
    KB_SIG_STATUS_PK_SMALL_ORDER = 6,    /* PublicKeySmallOrder    */
    KB_SIG_STATUS_MARSHALLING = 7,       /* MarshallingError: "invalid Ed25519 curve point" */
    KB_SIG_STATUS_INVALID = 8            /* InvalidSignature       */
} kb_sig_status;

/* flags for the scalar-multiplication entry points */
#define KB_FLAG_VARTIME 1u      /* scalars are public: direct table indexing instead of the
                                   reference's constant-time select (ge.rs:423-434,488-500) */
#define KB_FLAG_SHARED_POINT 2u /* `points` holds ONE 32-byte point used for every scalar  */

/* ---- context ---------------------------------------------------------------------- */
/* One context per device.  Creation builds the fixed-base tables on the device (about 8 ms): 48 KB for the constant-time
 * fixed-base multiplication and a 94 MB comb (15 positions x 2^16 multiples of B) shared by the verifiers and the
 * public-scalar multiplications.  Scratch grows with the largest batch seen (verify: 309 bytes per signature). */
int kb_ctx_create(int device, kb_ctx** out);
void kb_ctx_destroy(kb_ctx* ctx);
/* zero every device scratch buffer of the context (inputs such as secret scalars are staged there) */
int kb_ctx_wipe(kb_ctx* ctx);
const char* kb_last_error(const kb_ctx* ctx);
int kb_device_sm_count(const kb_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t kb_launch_count(const kb_ctx* ctx);
/* pinned host memory for callers that want full PCIe bandwidth on the kb_* copies */
void* kb_host_alloc(size_t bytes);
void kb_host_free(void* p);

/* ---- Point::mul (group/edwards25519/point.rs:207-225) ------------------------------- */
/* out[i] = compress(scalars[i] * B): Point::mul(s, None) -> ge_scalar_mult_base (ge.rs:442) */
int kb_point_mul_base_batch(kb_ctx* ctx, size_t n, const uint8_t* scalars, uint8_t* out, uint32_t flags);
/* out[i] = compress(scalars[i] * P_i): Point::mul(s, Some(p)) -> ge_scalar_mult (ge.rs:508).
 * status[i] = 1 when points[i] fails Point::unmarshal_binary (ge.rs:124; out[i] is then zero). */
int kb_point_mul_batch(kb_ctx* ctx, size_t n, const uint8_t* scalars, const uint8_t* points, uint8_t* out, uint8_t* status, uint32_t flags);

/* ---- encodings and point arithmetic ------------------------------------------------- */
/* Point::unmarshal_binary followed by marshal_binary (ge.rs:124-179 then :112-122):
 * out[i] = canonical re-encoding, status[i] = 1 if the input is not a curve point. */
int kb_point_recode_batch(kb_ctx* ctx, size_t n, const uint8_t* in, uint8_t* out, uint8_t* status);
/* The reference's serde/bincode wire format of a Point is its raw ExtendedGroupElement: X, Y, Z, T as
 * 10 signed 25.5-bit i32 limbs each (ge.rs:75-83, fe.rs:8) + a bool, unvalidated on decode (Deal::decode,
 * share/vss/pedersen/vss.rs:155-159).  limbs = n x 40 int32 (the bool stripped): out[i] = what
 * marshal_binary (ge.rs:112-122) returns for that element, for ANY limb values (Z = 0 gives 32 zero bytes). */
int kb_point_from_limbs_batch(kb_ctx* ctx, size_t n, const int32_t* limbs, uint8_t* out);
/* Point::add / Point::sub (point.rs:179,190) on encodings; status[i] = 1 if either fails to decode */
int kb_point_add_batch(kb_ctx* ctx, size_t n, const uint8_t* p, const uint8_t* q, uint8_t* out, uint8_t* status, int subtract);
/* ExtendedGroupElement::set_bytes (ge.rs:124-179) into the uncompressed device-friendly form used for chaining:
 * out128[i] = X, Y, Z, T as 4 x 8 little-endian 32-bit words (the form of kb_msm's partial128); status[i] = 1 and the
 * identity where the encoding does not decode. */
int kb_point_decompress_batch(kb_ctx* ctx, size_t n, const uint8_t* in, uint8_t* out128, uint8_t* status);
/* ExtendedGroupElement::write_bytes (ge.rs:112-122) from that form (any Z; one shared inversion per 8 points;
 * Z = 0 gives 32 zero bytes like the reference's fe_invert(0) = 0). */
int kb_point_compress_batch(kb_ctx* ctx, size_t n, const uint8_t* in128, uint8_t* out);
/* Point::eq (point.rs:227-241): equal_out[i] bit 0 = the two encodings decode to the same point (the reference
 * compares re-encodings, so a non-canonical y >= p equals its reduced twin); bit 1 = an operand does not decode. */
int kb_point_eq_batch(kb_ctx* ctx, size_t n, const uint8_t* p, const uint8_t* q, uint8_t* equal_out);
/* byte-level checks: bit0 = Point::is_canonical (point.rs:322, bug-compatible, SURVEY §A1),
 * bit1 = Point::has_small_order (point.rs:286), bit2 = decodes (ge.rs:124) */
int kb_point_check_batch(kb_ctx* ctx, size_t n, const uint8_t* in, uint8_t* flags_out);

/* ---- scalars -------------------------------------------------------------------------- */
/* Scalar::set_bytes on 64-byte digests (scalar.rs:175; integer_field/integer.rs:386): LE integer mod L */
int kb_sc_reduce64_batch(kb_ctx* ctx, size_t n, const uint8_t* in64, uint8_t* out32);
/* sc_mul_add (scalar.rs:279): out = (a*b + c) mod L; with c = 0 this is Scalar `*`, with b = 1 Scalar `+` */
int kb_sc_muladd_batch(kb_ctx* ctx, size_t n, const uint8_t* a, const uint8_t* b, const uint8_t* c, uint8_t* out);
/* Scalar::inv (scalar.rs:192-214): out = a^(L-2) mod L; Scalar::div(a, b) = a * inv(b) via kb_sc_muladd_batch */
int kb_sc_invert_batch(kb_ctx* ctx, size_t n, const uint8_t* a, uint8_t* out);
/* h_i = Scalar::set_bytes(SHA-512(R_i || A_i || M_i)) (eddsa_sig.rs:195-200, schnorr_sig.rs:128-141,
 * dss_sig.rs:312-326).  msg_off has n+1 entries; message i is msg[msg_off[i] .. msg_off[i+1]). */
int kb_challenge_batch(kb_ctx* ctx, size_t n, const uint8_t* r32, const uint8_t* a32, const uint8_t* msg, const uint64_t* msg_off, uint8_t* out32);

/* ---- signatures ----------------------------------------------------------------------- */
/* eddsa::verify_with_checks (sign/eddsa/eddsa_sig.rs:159-212); sig is n x 64 bytes.
 * Two independent kernel families return the reference's status: the default multiplies the reference's equation by
 * an odd u with u*h = v (mod 8L), |u|, |v| ~ 2^128 (128 doublings instead of 253; equivalent for every input because the
 * whole curve group has order 8L — csrc/half.cuh); KB_VERIFY_FULL=1 in the environment of kb_ctx_create selects the
 * full-length kernels.  KB_VERIFY_CHUNK=n / KB_VERIFY_CHUNK_LOG2=k cap the chunk size of the pipelined host-buffer calls. */
int kb_eddsa_verify_batch(kb_ctx* ctx, size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status);
/* schnorr::verify_with_checks (sign/schnorr/schnorr_sig.rs:53-110) */
int kb_schnorr_verify_batch(kb_ctx* ctx, size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status);

/* ---- key sets: verification under registered public keys ---------------------------------------------------- */
/* The signers of a DKG round, of DSS partial signatures or of a validator set are a small, fixed set of keys.  A key set
 * holds, per key, a comb over A from which h*A takes 32 table additions instead of a doubling loop, and every verify
 * call returns exactly what the general verifiers return for (keys[key_idx[i]], message i, sig[i]). */
typedef struct kb_keyset kb_keyset;
/* Registers nkeys public keys (32-byte encodings, exactly the bytes the verifiers would get as pk) with ctx.
 * Each key is checked once (Point::is_canonical incl. the §A1 quirk, has_small_order on bytes, decodes), and for
 * each key that passes, a comb kt[p][j] = (j+1)·2^(8p)·A, p = 0..31, j = 0..127, is built on the device
 * (affine (y+x, y-x, 2dxy), 96 B per entry: 384 KiB per key, in an allocation of the key set, not in scratch).
 * Keys that fail a check are accepted. Their signatures get the status the reference gives them.
 * KB_ERR_ARG for nkeys == 0 or a NULL pointer, KB_ERR_NOMEM if the tables do not fit.  A key set belongs to
 * its context (same device, errors in kb_last_error(ctx)) and must be destroyed before that context. */
int  kb_keyset_create(kb_ctx* ctx, size_t nkeys, const uint8_t* pk, kb_keyset** out);
void kb_keyset_destroy(kb_keyset* ks);
/* status[i] = what kb_eddsa_verify_batch (schnorr == 0) / kb_schnorr_verify_batch (schnorr != 0) returns for
 * (pk = keys[key_idx[i]], message i, sig[i]): same statuses and same check order.  msg / msg_off as in
 * kb_eddsa_verify_batch.  KB_ERR_ARG if any key_idx[i] >= nkeys (checked before anything is launched). */
int  kb_keyset_verify_batch(kb_keyset* ks, size_t n, const uint32_t* key_idx, const uint8_t* msg, const uint64_t* msg_off,
                            const uint8_t* sig, uint8_t* status, int schnorr);
/* device buffers + stream, ordered like every kb_dev_* call of the context.  An index >= nkeys gives status 0xFF
 * for that item, and the kernel reads nothing of the key set for it. */
int  kb_dev_keyset_verify(kb_keyset* ks, size_t n, const void* d_key_idx, const void* d_msg, const void* d_msg_off,
                          const void* d_sig, void* d_status, int schnorr, void* stream);
/* out[i] = compress(scalars[i] * keys[key_idx[i]]): Point::mul(s, Some(p)) with a registered p (point.rs:207,
 * ge.rs:508), the Diffie-Hellman step dh_exchange(secret, remote_public) (dh/dh_impl.rs:74-80) of encrypted_deal and
 * ECIES.  out and status are byte for byte what kb_point_mul_batch(ctx, n, scalars, keys[key_idx], out, status, flags)
 * returns, for every scalar (never reduced, also >= 2^255) and every key: status[i] = 1 and out[i] = 0 when the key does
 * not decode (status may be NULL).  A key with a comb needs no doublings: each of the 64 signed radix-16 windows selects
 * among 8 entries of its comb and adds once (constant-time select unless KB_FLAG_VARTIME); the other keys take the path
 * of kb_point_mul_batch.  The constant-time select reads 8 comb entries per window: with secret scalars under tens of
 * thousands of keys that traffic outweighs the saved work (DESIGN.md section 3.8).  flags: 0 or KB_FLAG_VARTIME, anything else is KB_ERR_ARG.  KB_ERR_ARG if any key_idx[i] >=
 * nkeys (checked before anything is launched).  Unless KB_FLAG_VARTIME is set, the scalars staged in device scratch
 * are zeroed before the call returns. */
int  kb_keyset_mul_batch(kb_keyset* ks, size_t n, const uint32_t* key_idx, const uint8_t* scalars, uint8_t* out,
                         uint8_t* status, uint32_t flags);
/* device buffers + stream, ordered like every kb_dev_* call of the context.  An index >= nkeys gives status 0xFF and
 * out[i] = 0 for that item, and the kernel reads nothing of the key set for it. */
int  kb_dev_keyset_mul(kb_keyset* ks, size_t n, const void* d_key_idx, const void* d_scalars, void* d_out, void* d_status,
                       uint32_t flags, void* stream);

/* EdDSA::sign (sign/eddsa/eddsa_sig.rs:120-152) for n (seed, message) pairs, with the key derivation of
 * Curve::new_key_and_seed_with_input (group/edwards25519/curve.rs:74-87): a = clamp(SHA-512(seed)[0..32]),
 * prefix = SHA-512(seed)[32..64], r = SHA-512(prefix || M) mod L, R = r*B, A = a*B, h = SHA-512(R || A || M) mod L,
 * s = (r + h*a) mod L.  sig[i] = R || s (64 bytes), pk[i] = A (may be NULL).  Deterministic: reproduces the
 * reference's golden signatures.  The secret scalars only meet the constant-time table select. */
int kb_eddsa_sign_batch(kb_ctx* ctx, size_t n, const uint8_t* seeds, const uint8_t* msg, const uint64_t* msg_off, uint8_t* sig, uint8_t* pk);

/* ---- committed polynomials (share/poly.rs) -------------------------------------------- */
/* PubPoly::eval (poly.rs:457-469) for npoly polynomials of t commitments each
 * (commits = npoly*t encodings, coefficient-major inside a polynomial):
 * out[k] = compress(poly[poly_id[k]].eval(idx[k])), status[k] = 1 if that polynomial holds an
 * undecodable commitment. */
int kb_pubpoly_eval_batch(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* commits, size_t m, const uint32_t* poly_id, const uint32_t* idx, uint8_t* out, uint8_t* status);
/* Group math of vss::pedersen Aggregator::verify_deal (share/vss/pedersen/vss.rs:899-912) and
 * PubPoly::check (poly.rs:526-530): verdict[k] = 1 iff shares[k]*B == poly[poly_id[k]].eval(idx[k])
 * on canonical bytes, 0 otherwise (including undecodable commitments). */
int kb_vss_verify_deals_batch(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* commits, size_t m, const uint32_t* poly_id, const uint32_t* idx, const uint8_t* shares, uint8_t* verdict);
/* A whole Pedersen-DKG deal-verification round (share/dkg/pedersen/dkg.rs:513-597 x n^2):
 * dealer d's polynomial is commits[d*t .. (d+1)*t), shares[d*n + i] is the share dealer d sent
 * to verifier i; verdict[d*n + i] as above.  Dealers [dealer_lo, dealer_hi) only — the unit a
 * rank owns when the round is sharded by dealer. */
int kb_dkg_verify_round(kb_ctx* ctx, size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, const uint8_t* commits, const uint8_t* shares, uint8_t* verdict);
/* The same round with the commitments in the reference's in-memory / serde form — X, Y, Z, T as 10 signed 25.5-bit i32
 * limbs each, 40 int32 per point (ge.rs:75-83; what a Rust caller holds in a PubPoly, so that it does not pay one field
 * inversion per commitment for marshal_binary).  The reference never validates that form (Deal::decode,
 * share/vss/pedersen/vss.rs:155-159); here a dealer with an element that is not a consistent representation of a curve
 * point (Z = 0, T Z != X Y, or off the curve) gets verdict 0 throughout. */
int kb_dkg_verify_round_limbs(kb_ctx* ctx, size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, const int32_t* commit_limbs, const uint8_t* shares, uint8_t* verdict);
/* PriPoly::eval (poly.rs:133-141) for npoly private polynomials of t coefficients at the indices 0..n-1:
 * out[d*n + i] = poly[d].eval(i) — the shares a dealer hands out (new_dealer, share/vss/pedersen/vss.rs:313). */
int kb_pripoly_eval_batch(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* coeffs, size_t n, uint8_t* out);
/* PubPoly::add (poly.rs:486-509): out[j] = a[j] + b[j] — kb_point_add_batch on t points.
 * dkg_key (share/dkg/pedersen/dkg.rs:905-954) folds PubPoly::add over all qualified dealers:
 * out[j] = sum_d commits[d*t + j], j < t; status[j] = 1 (and out[j] zero) if a commitment of column j is undecodable. */
int kb_pubpoly_sum(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* commits, uint8_t* out, uint8_t* status);

/* ---- protocol-level operations: the group math of the VSS / DKG / DSS verifiers as whole calls --------------------- */
/* How a caller hands over points that it holds as the reference's Point values. */
typedef enum kb_point_fmt {
    KB_POINT_ENC32 = 0,   /* 32-byte encodings (Point::marshal_binary, point.rs:35-41) */
    KB_POINT_LIMBS40 = 1  /* the in-memory / serde form: X, Y, Z, T as 10 signed 25.5-bit i32 limbs each (ge.rs:75-83) */
} kb_point_fmt;

/* session_id (share/vss/pedersen/vss.rs:1069-1090) for ndealers deals over the same verifier list:
 *   out32[d] = SHA-256( dealers[d] || verifiers[0..n) || commits[d*t .. (d+1)*t) || t as u32 LE )
 * over the points' canonical encodings (marshal_to), which are produced on the device (one shared inversion per 8 points —
 * the reference pays 1 + n + t inversions per call).  status[d] = 1 if a point that enters sid_d does not decode. */
int kb_vss_session_ids(kb_ctx* ctx, size_t ndealers, size_t n, size_t t, int fmt, const void* dealers, const void* verifiers, const void* commits, uint8_t* out32, uint8_t* status);
/* find_pub (share/dkg/pedersen/dkg.rs:1109-1116; the scan of new_verifier, share/vss/pedersen/vss.rs:541-550) for m queries
 * against one list: index_out[k] = smallest i with list[i] == queries[k] under Point::eq (canonical encodings), -1 if there
 * is none, -2 if the query does not decode.  The reference compresses both operands of every comparison. */
int kb_find_pub_batch(kb_ctx* ctx, size_t nlist, const void* list, size_t m, const void* queries, int fmt, int32_t* index_out);
/* One Pedersen-DKG deal-verification round for the dealers [dealer_lo, dealer_hi) as every verifier sees it
 * (share/dkg/pedersen/dkg.rs:513-597 process_deal, share/vss/pedersen/vss.rs:931-946 verify_response):
 *   verdict[d*n + i]      the share check of kb_dkg_verify_round (commits in `fmt`, whole arrays indexed by dealer)
 *   deal_status[k]        schnorr::verify of the dealer's signature on deal k        (dkg.rs:531)
 *   resp_status[k]        schnorr::verify of verifier i's signature on its response  (vss.rs:943)
 * where k = (d - dealer_lo)*n + i and the signature arrays (pk 32 B, sig 64 B, messages as flat bytes + n+1 offsets, the
 * layout of kb_schnorr_verify_batch) hold exactly the items of the dealer range.  A batch whose sig pointer is NULL is skipped. */
int kb_dkg_process_round(kb_ctx* ctx, size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, int fmt, const void* commits, const uint8_t* shares, uint8_t* verdict,
                         const uint8_t* deal_pk, const uint8_t* deal_msg, const uint64_t* deal_msg_off, const uint8_t* deal_sig, uint8_t* deal_status,
                         const uint8_t* resp_pk, const uint8_t* resp_msg, const uint64_t* resp_msg_off, const uint8_t* resp_sig, uint8_t* resp_status);
/* kb_dkg_process_round with the participants' keys registered as key sets: the signer of deal k is dealer
 * dealer_lo + k / n, key number dealer_lo + k / n of `dealers` (dealer keys are indexed by absolute dealer number, so a
 * rank that owns [dealer_lo, dealer_hi) passes the whole dealer set), and the signer of response k is verifier k % n, key
 * number k % n of `verifiers`.  verdict, deal_status and resp_status are exactly what kb_dkg_process_round returns for
 * those keys; the arrays are laid out as there, without the two pk arrays.  dealers and verifiers may be the same key set
 * (a new DKG: every participant deals and verifies) or two (resharing: old nodes deal, new nodes verify).
 * KB_ERR_ARG, before anything is launched, when dealers->nkeys < dealer_hi, verifiers->nkeys < n, a key set belongs to
 * another context, or a batch has a sig pointer but its key set is NULL.  A batch whose sig pointer is NULL is skipped.
 * Only msg[msg_off[0] .. msg_off[m]) of each batch is copied to the device. */
int kb_dkg_process_round_keyed(kb_ctx* ctx, const kb_keyset* dealers, const kb_keyset* verifiers,
                               size_t n, size_t t, size_t dealer_lo, size_t dealer_hi, int fmt, const void* commits, const uint8_t* shares, uint8_t* verdict,
                               const uint8_t* deal_msg, const uint64_t* deal_msg_off, const uint8_t* deal_sig, uint8_t* deal_status,
                               const uint8_t* resp_msg, const uint64_t* resp_msg_off, const uint8_t* resp_sig, uint8_t* resp_status);
/* vss::rabin verify_deal group math (share/vss/rabin/vss.rs:889-900): verdict[k] = 1 iff
 * f_shares[k]*G + g_shares[k]*H == poly[poly_id[k]].eval(idx[k]); H = derive_h(verifiers) supplied by the caller.
 * Both shares only meet constant-time table selects. */
int kb_vss_rabin_verify_deals_batch(kb_ctx* ctx, size_t npoly, size_t t, const uint8_t* commits, const uint8_t* h_point, size_t m, const uint32_t* poly_id, const uint32_t* idx,
                                    const uint8_t* f_shares, const uint8_t* g_shares, uint8_t* verdict);
/* DSS::process_partial_sig group math (sign/dss/dss_sig.rs:263-273) for m partial signatures of one signing session:
 *   hash = Scalar::set_bytes(SHA-512(random_commits[0] || long_commits[0] || msg))      (hash_sig, :312-326)
 *   verdict[k] = 1 iff partials[k]*B == random_poly.eval(idx[k]) + hash * long_poly.eval(idx[k])
 * in one chain of launches with the intermediate points kept uncompressed on the device.  hash_out32 (may be NULL) receives
 * hash.  The Schnorr check of the partial signature's own signature (:252) is kb_schnorr_verify_batch on the same batch. */
int kb_dss_verify_partials(kb_ctx* ctx, size_t t, const uint8_t* random_commits, const uint8_t* long_commits, const uint8_t* msg, size_t msg_len, size_t m, const uint32_t* idx, const uint8_t* partials,
                           uint8_t* verdict, uint8_t* hash_out32);
/* recover_commit (share/poly.rs:566-603) for ncols independent columns over the same k share indices idx (distinct):
 *   out[c] = sum_i lambda_i * points[c*k + i],   lambda_i = prod_{j!=i} x_j / prod_{j!=i} (x_j - x_i) mod L,  x = idx + 1
 * (the caller passes the first t shares in index order, xy_commit :535-562).  status[c] = 1 if a point of column c does
 * not decode. */
int kb_recover_commit_batch(kb_ctx* ctx, size_t ncols, size_t k, const uint32_t* idx, const uint8_t* points, uint8_t* out, uint8_t* status);
/* recover_pub_poly (share/poly.rs:607-635): the k commitments of the polynomial through the k public shares
 * (idx[j], points[j]):  out[c] = sum_j basis_j[c] * points[j] with the Lagrange basis polynomials of :640-671.  k <= 1023.
 * (The reference indexes its maps by position and therefore only works for idx = 0..k-1; any distinct indices are accepted here.) */
int kb_recover_pub_poly(kb_ctx* ctx, size_t k, const uint32_t* idx, const uint8_t* points, uint8_t* out, uint8_t* status);
/* resharing_key group math (share/dkg/pedersen/dkg.rs:996-1031): coeffs[i*new_t + c] = commitment c of the deal of the i-th
 * qualified old node (index idx[i]); out_commits[c] = recover_commit over column c; *check_out = pub_poly.check(share)
 * for the new share (share_idx, share32) — skipped when share32 or check_out is NULL. */
int kb_dkg_resharing_key(kb_ctx* ctx, size_t new_t, size_t k, const uint32_t* idx, const uint8_t* coeffs, uint32_t share_idx, const uint8_t* share32, uint8_t* out_commits, uint8_t* status, uint8_t* check_out);

/* ---- multi-scalar multiplication ------------------------------------------------------ */
/* out = compress(sum_i scalars[i] * P_i), the fold of Point::mul + Point::add (point.rs:179,207)
 * computed with Pippenger's bucket method.  *bad_points = number of undecodable inputs (the
 * result is then undefined).  partial128: if non-NULL, receives the UNcompressed sum as
 * 4 x 8 LE words (X,Y,Z,T) so that per-GPU partials can be combined with kb_point_sum. */
int kb_msm(kb_ctx* ctx, size_t n, const uint8_t* scalars, const uint8_t* points, uint8_t* out32, uint8_t* partial128, uint64_t* bad_points);
/* out = compress(sum of k uncompressed partials) — the final reduction after the NCCL gather */
int kb_point_sum(kb_ctx* ctx, size_t k, const uint8_t* partials128, uint8_t* out32);

/* ---- device-pointer variants (inputs already resident in HBM) --------------------------- */
/* d_msg_off: n+1 uint64 offsets in DEVICE memory.  The host-buffer calls validate the offsets (non-decreasing) and answer
 * KB_ERR_ARG; here they cannot be read by the host, so the caller must guarantee msg_off[i] <= msg_off[i+1] and
 * msg_off[n] <= the size of d_msg — a kernel that met a decreasing pair would read out of bounds. */
int kb_dev_eddsa_verify(kb_ctx* ctx, size_t n, const void* d_pk, const void* d_msg, const void* d_msg_off, const void* d_sig, void* d_status, int schnorr, void* stream);
int kb_dev_point_mul_base(kb_ctx* ctx, size_t n, const void* d_scalars, void* d_out, uint32_t flags, void* stream);
int kb_dev_point_mul(kb_ctx* ctx, size_t n, const void* d_scalars, const void* d_points, void* d_out, void* d_status, uint32_t flags, void* stream);
int kb_dev_msm(kb_ctx* ctx, size_t n, const void* d_scalars, const void* d_points, void* d_out32, void* d_partial128, void* d_bad_points, void* stream);
/* kb_dev_msm for points that are ALREADY DECODED: 128 bytes each, X, Y, Z, T as 4 x 8 little-endian words with any Z != 0
 * (the form of kb_point_decompress_batch, of partial128 and of every device-side producer): no decompression, the points
 * are made affine with one shared inversion per 8.  A point with Z = 0 or off the curve counts in *d_bad_points. */
int kb_dev_msm_ext(kb_ctx* ctx, size_t n, const void* d_scalars, const void* d_points128, void* d_out32, void* d_partial128, void* d_bad_points, void* stream);
int kb_dev_dkg_verify_round(kb_ctx* ctx, size_t n, size_t t, size_t ndealers, const void* d_commits, const void* d_shares, void* d_verdict, void* stream);
int kb_dev_dkg_verify_round_limbs(kb_ctx* ctx, size_t n, size_t t, size_t ndealers, const void* d_commit_limbs, const void* d_shares, void* d_verdict, void* stream);
int kb_dev_point_sum(kb_ctx* ctx, size_t k, const void* d_partials128, void* d_out32, void* stream);
/* the pure decompress (ExtendedGroupElement::set_bytes -> X, Y, Z, T words) and hash (SHA-512(R || A || M) mod L) stages */
int kb_dev_point_decompress(kb_ctx* ctx, size_t n, const void* d_in, void* d_out128, void* d_status, void* stream);
int kb_dev_challenge(kb_ctx* ctx, size_t n, const void* d_r32, const void* d_a32, const void* d_msg, const void* d_msg_off, void* d_out32, void* stream);
int kb_dev_pripoly_eval(kb_ctx* ctx, size_t npoly, size_t t, const void* d_coeffs, size_t n, void* d_out, void* stream);
/* kb_dkg_process_round on device buffers for ndealers dealers (arrays start at the first of them) */
int kb_dev_dkg_process_round(kb_ctx* ctx, size_t n, size_t t, size_t ndealers, int fmt, const void* d_commits, const void* d_shares, void* d_verdict,
                             const void* d_deal_pk, const void* d_deal_msg, const void* d_deal_msg_off, const void* d_deal_sig, void* d_deal_status,
                             const void* d_resp_pk, const void* d_resp_msg, const void* d_resp_msg_off, const void* d_resp_sig, void* d_resp_status, void* stream);
/* kb_dkg_process_round_keyed on device buffers for the ndealers dealers from dealer_lo on (the arrays start at the first of
 * them; dealer keys are still indexed by absolute dealer number): the checks of the host form with dealer_hi =
 * dealer_lo + ndealers, then ordered like every kb_dev_* call of the context. */
int kb_dev_dkg_process_round_keyed(kb_ctx* ctx, const kb_keyset* dealers, const kb_keyset* verifiers,
                                   size_t n, size_t t, size_t dealer_lo, size_t ndealers, int fmt, const void* d_commits, const void* d_shares, void* d_verdict,
                                   const void* d_deal_msg, const void* d_deal_msg_off, const void* d_deal_sig, void* d_deal_status,
                                   const void* d_resp_msg, const void* d_resp_msg_off, const void* d_resp_sig, void* d_resp_status, void* stream);

/* ---- multi-device context: ONE host batch sharded over the GPUs of a box, from one process ---------------------------
 * (SURVEY §8b/§8e).  kb_mctx_create builds one kb_ctx per listed device and, for more than one device, an NCCL communicator
 * over them (libnccl.so.2 is bound at run time; KB_NCCL_LIB overrides the name).  Every call takes ordinary HOST buffers
 * holding the WHOLE batch and returns the WHOLE result:
 *   signatures, scalar multiplications   split by index      — no exchange between devices
 *   DKG rounds                           split by dealer     — no exchange between devices
 *   MSM                                  split by points     — each device reduces its points to one 128-byte partial,
 *                                        ncclAllGather of the partials over NVLink, every device folds them (the only
 *                                        data-path collective there is)
 * One host thread per device drives it, so the shards' copies run concurrently.  A kb_mctx is not thread-safe. */
#define KB_MAX_DEVICES 16
typedef struct kb_mctx kb_mctx;
int kb_mctx_create(const int* devices, int ndev, kb_mctx** out);
void kb_mctx_destroy(kb_mctx* m);
int kb_mctx_device_count(const kb_mctx* m);
kb_ctx* kb_mctx_ctx(kb_mctx* m, int i);   /* the single-device context of the i-th device (owned by m) */
const char* kb_mctx_last_error(const kb_mctx* m);
uint64_t kb_mctx_launch_count(const kb_mctx* m);
/* kb_eddsa_verify_batch / kb_schnorr_verify_batch (schnorr != 0) over all devices */
int kb_mctx_verify_batch(kb_mctx* m, size_t n, const uint8_t* pk, const uint8_t* msg, const uint64_t* msg_off, const uint8_t* sig, uint8_t* status, int schnorr);
int kb_mctx_point_mul_base_batch(kb_mctx* m, size_t n, const uint8_t* scalars, uint8_t* out, uint32_t flags);
int kb_mctx_point_mul_batch(kb_mctx* m, size_t n, const uint8_t* scalars, const uint8_t* points, uint8_t* out, uint8_t* status, uint32_t flags);
/* kb_dkg_verify_round / kb_dkg_process_round for ndealers dealers (all arrays whole: commitments and shares by dealer,
 * the signature arrays with one item per (dealer, verifier), k = d*n + i) */
int kb_mctx_dkg_verify_round(kb_mctx* m, size_t n, size_t t, size_t ndealers, int fmt, const void* commits, const uint8_t* shares, uint8_t* verdict);
int kb_mctx_dkg_process_round(kb_mctx* m, size_t n, size_t t, size_t ndealers, int fmt, const void* commits, const uint8_t* shares, uint8_t* verdict,
                              const uint8_t* deal_pk, const uint8_t* deal_msg, const uint64_t* deal_msg_off, const uint8_t* deal_sig, uint8_t* deal_status,
                              const uint8_t* resp_pk, const uint8_t* resp_msg, const uint64_t* resp_msg_off, const uint8_t* resp_sig, uint8_t* resp_status);
/* Key sets over all devices.  A kb_mkeyset holds one kb_keyset per device, and each of them holds EVERY key: the keys are
 * replicated, not sharded, so a key set of K keys takes 384 KiB x K of memory on each GPU.  kb_mctx_keyset_create builds
 * the combs of all devices concurrently; if one device fails, the sets already built are destroyed and the error is in
 * kb_mctx_last_error.  A kb_mkeyset must be destroyed before its kb_mctx. */
typedef struct kb_mkeyset kb_mkeyset;
int  kb_mctx_keyset_create(kb_mctx* m, size_t nkeys, const uint8_t* pk, kb_mkeyset** out);
void kb_mctx_keyset_destroy(kb_mkeyset* ks);
/* kb_keyset_verify_batch split by index over all devices.  Every key index is checked before any device starts
 * (KB_ERR_ARG); each device copies only the message bytes of its own items. */
int  kb_mctx_keyset_verify_batch(kb_mkeyset* ks, size_t n, const uint32_t* key_idx, const uint8_t* msg, const uint64_t* msg_off,
                                 const uint8_t* sig, uint8_t* status, int schnorr);
/* kb_keyset_mul_batch split by index over all devices, each against its own copy of the key set.  Flags and every key
 * index are checked before any device starts (KB_ERR_ARG). */
int  kb_mctx_keyset_mul_batch(kb_mkeyset* ks, size_t n, const uint32_t* key_idx, const uint8_t* scalars, uint8_t* out,
                              uint8_t* status, uint32_t flags);
/* kb_dkg_process_round_keyed for ndealers dealers split by dealer (arrays whole, as kb_mctx_dkg_process_round has them):
 * each device runs its dealer range against its own copy of the key sets. */
int  kb_mctx_dkg_process_round_keyed(kb_mctx* m, const kb_mkeyset* dealers, const kb_mkeyset* verifiers, size_t n, size_t t, size_t ndealers, int fmt,
                                     const void* commits, const uint8_t* shares, uint8_t* verdict,
                                     const uint8_t* deal_msg, const uint64_t* deal_msg_off, const uint8_t* deal_sig, uint8_t* deal_status,
                                     const uint8_t* resp_msg, const uint64_t* resp_msg_off, const uint8_t* resp_sig, uint8_t* resp_status);
/* kb_msm over all devices */
int kb_mctx_msm(kb_mctx* m, size_t n, const uint8_t* scalars, const uint8_t* points, uint8_t* out32, uint64_t* bad_points);

/* ---- measurement ---------------------------------------------------------------------- */
/* Integer-multiply roofline probe: runs `iters` dependent-chain-free IMAD.WIDE.U32 per thread
 * on every SM and returns the achieved 32x32->64 multiply-accumulates per second.
 * kind: 0 = IMAD.WIDE.U32 (64-bit accumulate, nothing else in the loop), 1 = IMAD (32-bit lo), 2 = IMAD.WIDE.U32.X carry chains,
 * 3 = the library's own fe_mul (reported in IMAD-eq at 72 per multiplication). */
int kb_probe_imad(kb_ctx* ctx, int kind, int iters, double* macs_per_sec, double* elapsed_ms);
/* Per-kernel timing of the verifiers.  enable = 1/0 switches CUDA-event recording (on the launch stream, around
 * each of the two launches of a verify call) on or off; with ms_out != NULL the call then waits for the most recent
 * kb_dev_eddsa_verify and returns ms_out[0] = first launch (k_verify_half_prep / k_verify_stage1), ms_out[1] =
 * second launch (k_verify_half_main / k_verify_stage2).  This is how bench.py times the dominant kernel live. */
int kb_verify_kernel_times(kb_ctx* ctx, int enable, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* KYBER_B200_H */
