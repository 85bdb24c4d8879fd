//! Batch entry points behind kyber-rs's existing trait surface (src/group.rs: `Point` :85,
//! `Scalar` :22).  NOT COMPILED in the environment this repository is built in.
//!
//! Protocol code keeps using `Group`/`Point`/`Scalar`; where it loops over `Point::mul`,
//! `PubPoly::check` or `schnorr::verify` today it can hand the whole loop to one call here and
//! gets, item by item, exactly what the scalar call would have returned (compressed encodings,
//! `SignatureError` variants) — that bit-exactness is what `tests/` checks through the same C ABI.
use kyber_b200_sys as sys;
use kyber_rs::encoding::{BinaryMarshaler, BinaryUnmarshaler, MarshallingError};
use kyber_rs::group::edwards25519::{Point as EdPoint, Scalar as EdScalar};
use kyber_rs::share::poly::{PriShare, PubPoly};
use kyber_rs::sign::error::SignatureError;

#[derive(Debug)]
pub enum GpuError {
    Arg,
    Cuda(String),
    NoMem,
    /// an input point does not decode (what `Point::unmarshal_binary` reports as MarshallingError::InvalidInput);
    /// the index of the first such item
    InvalidPoint(usize),
}

/// How a DKG round checks its shares (`kb_round_check`).
#[derive(Clone, Copy, PartialEq, Eq, Debug)]
pub enum RoundCheck {
    /// every share is evaluated (the default)
    Exact,
    /// one random linear combination per dealer; dealers that fail it are checked share by share.  The verdicts are the
    /// exact ones except with probability at most 2^-128 per dealer with a wrong share.
    Batched,
}

/// One CUDA device, one host thread — kyber-rs itself is single-threaded (SURVEY §8b).
pub struct Gpu {
    ctx: *mut sys::kb_ctx,
}

impl Gpu {
    pub fn new(device: i32) -> Result<Self, GpuError> {
        let mut ctx = std::ptr::null_mut();
        match unsafe { sys::kb_ctx_create(device, &mut ctx) } {
            sys::KB_OK => Ok(Gpu { ctx }),
            sys::KB_ERR_NOMEM => Err(GpuError::NoMem),
            _ => Err(GpuError::Cuda("no usable CUDA device (there is no CPU fallback)".into())),
        }
    }
    /// How the DKG rounds of this context check their shares (`kb_ctx_set_round_check`); a new context is `Exact`.
    pub fn set_round_check(&self, mode: RoundCheck) -> Result<(), GpuError> {
        let m = match mode {
            RoundCheck::Exact => 0,
            RoundCheck::Batched => 1,
        };
        self.check(unsafe { sys::kb_ctx_set_round_check(self.ctx, m) })
    }
    /// Dealers the last round call checked share by share (0 after an `Exact` round).
    pub fn round_fallbacks(&self) -> Result<u64, GpuError> {
        let mut d = 0u64;
        self.check(unsafe { sys::kb_ctx_round_fallbacks(self.ctx, &mut d) })?;
        Ok(d)
    }
    /// The share checks participants `ver_lo..ver_hi` run in `process_deal` (share/dkg/pedersen/dkg.rs:513-597), for every
    /// dealer in one call: `polys[d]` is dealer `d`'s committed polynomial and `shares[d * k + c]` the share it sent to
    /// verifier `ver_lo + c`, `k = ver_hi - ver_lo` (`k = 1` for one node).  `verdict[d * k + c]` is what
    /// `Aggregator::verify_deal` (vss.rs:899-912) decides; exact in both round-check modes.
    pub fn dkg_verify_columns(&self, n: usize, polys: &[Vec<EdPoint>], ver_lo: usize, ver_hi: usize, shares: &[EdScalar]) -> Result<Vec<bool>, GpuError> {
        let t = polys.first().map(|p| p.len()).unwrap_or(0);
        let k = ver_hi.saturating_sub(ver_lo);
        assert!(polys.iter().all(|p| p.len() == t) && shares.len() == polys.len() * k);
        let limbs: Vec<i32> = polys.iter().flat_map(|p| pack_point_limbs(p)).collect();
        let sh = pack_scalars(shares);
        let mut verdict = vec![0u8; shares.len()];
        self.check(unsafe { sys::kb_dkg_verify_columns(self.ctx, n, t, 0, polys.len(), ver_lo, ver_hi, 1, limbs.as_ptr().cast(), sh.as_ptr(), verdict.as_mut_ptr()) })?;
        Ok(verdict.into_iter().map(|v| v == 1).collect())
    }
    fn check(&self, rc: i32) -> Result<(), GpuError> {
        match rc {
            sys::KB_OK => Ok(()),
            sys::KB_ERR_ARG => Err(GpuError::Arg),
            sys::KB_ERR_NOMEM => Err(GpuError::NoMem),
            _ => Err(GpuError::Cuda(unsafe { std::ffi::CStr::from_ptr(sys::kb_last_error(self.ctx)) }.to_string_lossy().into_owned())),
        }
    }
}
impl Drop for Gpu {
    fn drop(&mut self) {
        unsafe { sys::kb_ctx_destroy(self.ctx) }
    }
}

fn pack_scalars(s: &[EdScalar]) -> Vec<u8> {
    s.iter().flat_map(|x| x.v).collect() // Scalar.v: [u8; 32], raw (scalar.rs:24)
}
fn pack_points(p: &[EdPoint]) -> Vec<u8> {
    p.iter().flat_map(|x| x.marshal_binary().expect("32 bytes")).collect()
}
/// The in-memory form of a `Point` (ge.rs:75-83: X, Y, Z, T as 10 i32 limbs each) — what the `_limbs` / `KB_POINT_LIMBS40`
/// entry points take, so that a caller holding thousands of commitments does not pay one field inversion each for
/// `marshal_binary` (SURVEY §8f-3).
fn pack_point_limbs(p: &[EdPoint]) -> Vec<i32> {
    p.iter().flat_map(|x| x.ge_mut_ref_limbs()).collect() // accessor to be added next to Point::ge (point.rs:24)
}
fn unpack_points(b: &[u8]) -> Vec<EdPoint> {
    b.chunks(32)
        .map(|c| {
            let mut p = EdPoint::default();
            p.unmarshal_binary(c).expect("library output is a canonical encoding");
            p
        })
        .collect()
}

/// Batch companion of `group::Point::mul` (group.rs:139; point.rs:207-225).
pub trait BatchPoint: Sized {
    /// `points = None` multiplies the standard base (ge_scalar_mult_base, ge.rs:442).
    fn mul_batch(gpu: &Gpu, scalars: &[EdScalar], points: Option<&[Self]>) -> Result<Vec<Self>, GpuError>;
}
impl BatchPoint for EdPoint {
    fn mul_batch(gpu: &Gpu, scalars: &[EdScalar], points: Option<&[EdPoint]>) -> Result<Vec<EdPoint>, GpuError> {
        let n = scalars.len();
        let s = pack_scalars(scalars);
        let mut out = vec![0u8; 32 * n];
        match points {
            None => gpu.check(unsafe { sys::kb_point_mul_base_batch(gpu.ctx, n, s.as_ptr(), out.as_mut_ptr(), 0) })?,
            Some(ps) => {
                assert_eq!(ps.len(), n);
                let p = pack_points(ps);
                let mut st = vec![0u8; n];
                gpu.check(unsafe { sys::kb_point_mul_batch(gpu.ctx, n, s.as_ptr(), p.as_ptr(), out.as_mut_ptr(), st.as_mut_ptr(), 0) })?;
                // an undecodable input leaves 32 zero bytes, which would decode as a valid order-4 point: report it instead
                if let Some(i) = st.iter().position(|&x| x != 0) {
                    return Err(GpuError::InvalidPoint(i));
                }
            }
        }
        Ok(unpack_points(&out))
    }
}

fn status_to_result(st: u8) -> Result<(), SignatureError> {
    match st {
        0 => Ok(()),
        1 => Err(SignatureError::InvalidSignatureLength("expect 64".to_owned())),
        2 => Err(SignatureError::SignatureNotCanonical),
        3 => Err(SignatureError::RNotCanonical),
        4 => Err(SignatureError::RSmallOrder),
        5 => Err(SignatureError::PublicKeyNotCanonical),
        6 => Err(SignatureError::PublicKeySmallOrder),
        7 => Err(SignatureError::MarshallingError(MarshallingError::InvalidInput("invalid Ed25519 curve point".to_owned()))),
        _ => Err(SignatureError::InvalidSignature("reconstructed S is not equal to signature".to_owned())),
    }
}

/// Batch companion of `eddsa::verify_with_checks` (sign/eddsa/eddsa_sig.rs:159-212) and, with
/// `schnorr = true`, of `schnorr::verify_with_checks` (sign/schnorr/schnorr_sig.rs:53-110).
/// Items are (public key bytes, message, signature).
pub fn verify_batch(gpu: &Gpu, items: &[(&[u8], &[u8], &[u8])], schnorr: bool) -> Result<Vec<Result<(), SignatureError>>, GpuError> {
    let mut res: Vec<Option<Result<(), SignatureError>>> = vec![None; items.len()];
    let (mut pk, mut sig, mut msg, mut off, mut idx) = (vec![], vec![], vec![], vec![0u64], vec![]);
    for (i, (p, m, s)) in items.iter().enumerate() {
        if s.len() != 64 {
            res[i] = Some(status_to_result(1)); // eddsa_sig.rs:161 / schnorr_sig.rs:68
            continue;
        }
        if p.len() != 32 {
            // the reference cannot even build such a key: unmarshal_binary fails; one wrong-length key must not
            // misalign every later item of the packed batch
            res[i] = Some(status_to_result(5));
            continue;
        }
        pk.extend_from_slice(p);
        sig.extend_from_slice(s);
        msg.extend_from_slice(m);
        off.push(msg.len() as u64);
        idx.push(i);
    }
    let n = idx.len();
    let mut st = vec![0u8; n];
    let f = if schnorr { sys::kb_schnorr_verify_batch } else { sys::kb_eddsa_verify_batch };
    gpu.check(unsafe { f(gpu.ctx, n, pk.as_ptr(), msg.as_ptr(), off.as_ptr(), sig.as_ptr(), st.as_mut_ptr()) })?;
    for (k, i) in idx.into_iter().enumerate() {
        res[i] = Some(status_to_result(st[k]));
    }
    Ok(res.into_iter().map(|r| r.unwrap()).collect())
}

/// Public keys registered once with a `Gpu` — the dealers of a DKG round, the participants of a DSS session, a validator
/// set — so that their signatures are verified by key index without decompressing the key or doubling per signature.
/// Item by item the result is what `verify_batch` returns for the same key bytes.  Borrows the `Gpu`: a key set is
/// dropped before its context.
pub struct KeySet<'a> {
    gpu: &'a Gpu,
    ks: *mut sys::kb_keyset,
    nkeys: usize,
}

impl<'a> KeySet<'a> {
    /// Registers `keys` (32-byte encodings, the bytes a verifier would get as the public key).  Keys that fail the
    /// reference's checks are accepted; their signatures get the reference's error.  384 KiB of device memory per key.
    pub fn new(gpu: &'a Gpu, keys: &[[u8; 32]]) -> Result<Self, GpuError> {
        let flat: Vec<u8> = keys.iter().flat_map(|k| k.iter().copied()).collect();
        let mut ks = std::ptr::null_mut();
        gpu.check(unsafe { sys::kb_keyset_create(gpu.ctx, keys.len(), flat.as_ptr(), &mut ks) })?;
        Ok(KeySet { gpu, ks, nkeys: keys.len() })
    }
    /// Items are (key index, message, signature); `schnorr` selects `schnorr::verify_with_checks` instead of
    /// `eddsa::verify_with_checks`.  A key index outside the set is `GpuError::Arg`.
    pub fn verify_batch(&self, items: &[(u32, &[u8], &[u8])], schnorr: bool) -> Result<Vec<Result<(), SignatureError>>, GpuError> {
        if items.iter().any(|(k, _, _)| *k as usize >= self.nkeys) {
            return Err(GpuError::Arg);
        }
        let mut res: Vec<Option<Result<(), SignatureError>>> = vec![None; items.len()];
        let (mut key_idx, mut sig, mut msg, mut off, mut idx) = (vec![], vec![], vec![], vec![0u64], vec![]);
        for (i, (k, m, s)) in items.iter().enumerate() {
            if s.len() != 64 {
                res[i] = Some(status_to_result(1)); // eddsa_sig.rs:161 / schnorr_sig.rs:68
                continue;
            }
            key_idx.push(*k);
            sig.extend_from_slice(s);
            msg.extend_from_slice(m);
            off.push(msg.len() as u64);
            idx.push(i);
        }
        let n = idx.len();
        let mut st = vec![0u8; n];
        self.gpu.check(unsafe { sys::kb_keyset_verify_batch(self.ks, n, key_idx.as_ptr(), msg.as_ptr(), off.as_ptr(), sig.as_ptr(), st.as_mut_ptr(), schnorr as i32) })?;
        for (k, i) in idx.into_iter().enumerate() {
            res[i] = Some(status_to_result(st[k]));
        }
        Ok(res.into_iter().map(|r| r.unwrap()).collect())
    }
    /// Items are (public key bytes, message, signature), as `verify_batch` takes them, with the same result item by item:
    /// an item whose 32 key bytes equal a registered key's is verified from that key's comb, every other item by the
    /// general verifier, in one call.  Also returns how many items took the comb path.
    pub fn verify_pk_batch(&self, items: &[(&[u8], &[u8], &[u8])], schnorr: bool) -> Result<(Vec<Result<(), SignatureError>>, u64), GpuError> {
        let mut res: Vec<Option<Result<(), SignatureError>>> = vec![None; items.len()];
        let (mut pk, mut sig, mut msg, mut off, mut idx) = (vec![], vec![], vec![], vec![0u64], vec![]);
        for (i, (p, m, s)) in items.iter().enumerate() {
            if s.len() != 64 {
                res[i] = Some(status_to_result(1)); // eddsa_sig.rs:161 / schnorr_sig.rs:68
                continue;
            }
            if p.len() != 32 {
                res[i] = Some(status_to_result(5)); // as verify_batch: the reference cannot build such a key
                continue;
            }
            pk.extend_from_slice(p);
            sig.extend_from_slice(s);
            msg.extend_from_slice(m);
            off.push(msg.len() as u64);
            idx.push(i);
        }
        let n = idx.len();
        let mut st = vec![0u8; n];
        let mut hits = 0u64;
        self.gpu.check(unsafe { sys::kb_keyset_verify_pk_batch(self.ks, n, pk.as_ptr(), msg.as_ptr(), off.as_ptr(), sig.as_ptr(), st.as_mut_ptr(), schnorr as i32, &mut hits) })?;
        for (k, i) in idx.into_iter().enumerate() {
            res[i] = Some(status_to_result(st[k]));
        }
        Ok((res.into_iter().map(|r| r.unwrap()).collect(), hits))
    }
    /// Batch companion of `Point::mul(s, Some(pk))` for registered keys — the `dh_exchange(secret, remote_public)` step
    /// (dh/dh_impl.rs:74-80) of `encrypted_deal` and ECIES.  Items are (key index, scalar); the result is what
    /// `BatchPoint::mul_batch` returns for the same key bytes, from the keys' combs.  The scalars are secret: the table
    /// select is constant-time.  A key index outside the set is `GpuError::Arg`, a key that does not decode
    /// `GpuError::InvalidPoint`.
    pub fn mul_batch(&self, items: &[(u32, EdScalar)]) -> Result<Vec<EdPoint>, GpuError> {
        if items.iter().any(|(k, _)| *k as usize >= self.nkeys) {
            return Err(GpuError::Arg);
        }
        let n = items.len();
        let key_idx: Vec<u32> = items.iter().map(|(k, _)| *k).collect();
        let scalars: Vec<EdScalar> = items.iter().map(|(_, s)| s.clone()).collect();
        let s = pack_scalars(&scalars);
        let mut out = vec![0u8; 32 * n];
        let mut st = vec![0u8; n];
        self.gpu.check(unsafe { sys::kb_keyset_mul_batch(self.ks, n, key_idx.as_ptr(), s.as_ptr(), out.as_mut_ptr(), st.as_mut_ptr(), 0) })?;
        if let Some(i) = st.iter().position(|&x| x != 0) {
            return Err(GpuError::InvalidPoint(i));
        }
        Ok(unpack_points(&out))
    }
}
impl Drop for KeySet<'_> {
    fn drop(&mut self) {
        unsafe { sys::kb_keyset_destroy(self.ks) }
    }
}

/// Batch companion of `schnorr::sign` (sign/schnorr/schnorr_sig.rs:25-47).  Items are (secret x, nonce k, message); the
/// reference draws k from its random stream, here the caller supplies it (the library cannot detect a reused nonce, and
/// a nonce used twice under one key reveals that key).  Returns the 64-byte signatures R || s and the public keys x*B.
pub fn schnorr_sign_batch(gpu: &Gpu, items: &[(EdScalar, EdScalar, &[u8])]) -> Result<(Vec<[u8; 64]>, Vec<EdPoint>), GpuError> {
    let n = items.len();
    let x = pack_scalars(&items.iter().map(|(x, _, _)| x.clone()).collect::<Vec<_>>());
    let k = pack_scalars(&items.iter().map(|(_, k, _)| k.clone()).collect::<Vec<_>>());
    let (msg, off) = pack_messages(items.iter().map(|(_, _, m)| *m));
    let mut sig = vec![0u8; 64 * n];
    let mut pk = vec![0u8; 32 * n];
    gpu.check(unsafe { sys::kb_schnorr_sign_batch(gpu.ctx, n, x.as_ptr(), k.as_ptr(), msg.as_ptr(), off.as_ptr(), sig.as_mut_ptr(), pk.as_mut_ptr()) })?;
    Ok((unpack_sigs(&sig), unpack_points(&pk)))
}

fn pack_messages<'m>(msgs: impl Iterator<Item = &'m [u8]>) -> (Vec<u8>, Vec<u64>) {
    let (mut msg, mut off) = (vec![], vec![0u64]);
    for m in msgs {
        msg.extend_from_slice(m);
        off.push(msg.len() as u64);
    }
    (msg, off)
}
fn unpack_sigs(b: &[u8]) -> Vec<[u8; 64]> {
    b.chunks(64).map(|c| c.try_into().expect("64 bytes")).collect()
}

/// Which signing function a `SignerSet` serves.
#[derive(Clone, Copy, PartialEq, Eq, Debug)]
pub enum SignerKind {
    /// keys are secret scalars x; `schnorr::sign` (schnorr_sig.rs:25-47), nonces from the caller
    Schnorr,
    /// keys are 32-byte seeds; `EdDSA::sign` (eddsa_sig.rs:120-152) with the key derivation of curve.rs:74-87,
    /// deterministic nonces
    EdDSA,
}

/// Secret keys registered once with a `Gpu` — the key each participant of a DKG round signs its deals and responses
/// with — so that a signature pays one constant-time fixed-base multiplication instead of two.  Signatures are byte for
/// byte those of `schnorr_sign_batch` / `kb_eddsa_sign_batch` under the same key.  Borrows the `Gpu`: a signer set is
/// dropped before its context; dropping it zeroes the keys on the device.
pub struct SignerSet<'a> {
    gpu: &'a Gpu,
    ss: *mut sys::kb_signerset,
    nkeys: usize,
    kind: SignerKind,
    /// the public key of each registered key (x*B or a*B)
    pub public: Vec<EdPoint>,
}

impl<'a> SignerSet<'a> {
    /// Registers `keys`: secret scalars (`SignerKind::Schnorr`, their raw 32 bytes) or seeds (`SignerKind::EdDSA`).
    pub fn new(gpu: &'a Gpu, keys: &[[u8; 32]], kind: SignerKind) -> Result<Self, GpuError> {
        let flat: Vec<u8> = keys.iter().flat_map(|k| k.iter().copied()).collect();
        let mut pk = vec![0u8; 32 * keys.len()];
        let mut ss = std::ptr::null_mut();
        let k = if kind == SignerKind::EdDSA { sys::KB_SIGNER_EDDSA } else { sys::KB_SIGNER_SCHNORR };
        gpu.check(unsafe { sys::kb_signerset_create(gpu.ctx, keys.len(), flat.as_ptr(), k, pk.as_mut_ptr(), &mut ss) })?;
        Ok(SignerSet { gpu, ss, nkeys: keys.len(), kind, public: unpack_points(&pk) })
    }
    /// Items are (key index, message); `nonces` holds one nonce per item for a Schnorr set and must be `None` for an
    /// EdDSA set.  A key index outside the set or the other nonce / kind combination is `GpuError::Arg`.
    pub fn sign_batch(&self, items: &[(u32, &[u8])], nonces: Option<&[EdScalar]>) -> Result<Vec<[u8; 64]>, GpuError> {
        let n = items.len();
        if items.iter().any(|(k, _)| *k as usize >= self.nkeys) || (self.kind == SignerKind::Schnorr) != nonces.is_some() || nonces.map_or(false, |k| k.len() != n) {
            return Err(GpuError::Arg);
        }
        let key_idx: Vec<u32> = items.iter().map(|(k, _)| *k).collect();
        let (msg, off) = pack_messages(items.iter().map(|(_, m)| *m));
        let k = nonces.map(pack_scalars);
        let mut sig = vec![0u8; 64 * n];
        let kp = k.as_ref().map_or(std::ptr::null(), |v| v.as_ptr());
        self.gpu.check(unsafe { sys::kb_signerset_sign_batch(self.ss, n, key_idx.as_ptr(), kp, msg.as_ptr(), off.as_ptr(), sig.as_mut_ptr()) })?;
        Ok(unpack_sigs(&sig))
    }
}
impl Drop for SignerSet<'_> {
    fn drop(&mut self) {
        unsafe { sys::kb_signerset_destroy(self.ss) }
    }
}

/// Batch companion of `PubPoly::eval` / `PubPoly::check` (share/poly.rs:457-469, :526-530) — the
/// group math of `Aggregator::verify_deal` (share/vss/pedersen/vss.rs:899-912).
pub trait PubPolyBatch {
    fn eval_batch(&self, gpu: &Gpu, idx: &[u32]) -> Result<Vec<EdPoint>, GpuError>;
    fn check_batch(&self, gpu: &Gpu, shares: &[PriShare<EdScalar>]) -> Result<Vec<bool>, GpuError>;
}
impl<G: kyber_rs::Group<POINT = EdPoint>> PubPolyBatch for PubPoly<G> {
    fn eval_batch(&self, gpu: &Gpu, idx: &[u32]) -> Result<Vec<EdPoint>, GpuError> {
        let (_, commits) = self.info();
        let c = pack_points(&commits);
        let pid = vec![0u32; idx.len()];
        let mut out = vec![0u8; 32 * idx.len()];
        let mut st = vec![0u8; idx.len()];
        gpu.check(unsafe { sys::kb_pubpoly_eval_batch(gpu.ctx, 1, commits.len(), c.as_ptr(), idx.len(), pid.as_ptr(), idx.as_ptr(), out.as_mut_ptr(), st.as_mut_ptr()) })?;
        if let Some(i) = st.iter().position(|&x| x != 0) {
            return Err(GpuError::InvalidPoint(i));
        }
        Ok(unpack_points(&out))
    }
    fn check_batch(&self, gpu: &Gpu, shares: &[PriShare<EdScalar>]) -> Result<Vec<bool>, GpuError> {
        let (_, commits) = self.info();
        let c = pack_points(&commits);
        let idx: Vec<u32> = shares.iter().map(|s| s.i as u32).collect();
        let pid = vec![0u32; idx.len()];
        let sh: Vec<u8> = shares.iter().flat_map(|s| s.v.v).collect();
        let mut verdict = vec![0u8; idx.len()];
        gpu.check(unsafe { sys::kb_vss_verify_deals_batch(gpu.ctx, 1, commits.len(), c.as_ptr(), idx.len(), pid.as_ptr(), idx.as_ptr(), sh.as_ptr(), verdict.as_mut_ptr()) })?;
        Ok(verdict.into_iter().map(|v| v == 1).collect())
    }
}

/// `sum_i s_i * P_i` — what `PriPoly::commit` / `recover_commit` (share/poly.rs:195, :566) fold by hand.
pub fn msm(gpu: &Gpu, scalars: &[EdScalar], points: &[EdPoint]) -> Result<EdPoint, GpuError> {
    assert_eq!(scalars.len(), points.len());
    let (s, p) = (pack_scalars(scalars), pack_points(points));
    let mut out = [0u8; 32];
    let mut bad = 0u64;
    gpu.check(unsafe { sys::kb_msm(gpu.ctx, scalars.len(), s.as_ptr(), p.as_ptr(), out.as_mut_ptr(), std::ptr::null_mut(), &mut bad) })?;
    if bad != 0 {
        return Err(GpuError::InvalidPoint(0)); // the sum is undefined when an input does not decode
    }
    Ok(unpack_points(&out).remove(0))
}


/// One DKG deal-verification round for this node's view of `dealers` (share/dkg/pedersen/dkg.rs:513-597): every dealer's
/// committed polynomial against the share it sent to every verifier, the commitments handed over in their in-memory form
/// (no per-commitment `marshal_binary`).  `verdict[d * n + i]` is what `Aggregator::verify_deal` (vss.rs:899-912) decides.
pub fn dkg_verify_round(gpu: &Gpu, n: usize, polys: &[Vec<EdPoint>], shares: &[EdScalar]) -> Result<Vec<bool>, GpuError> {
    let t = polys.first().map(|p| p.len()).unwrap_or(0);
    assert!(polys.iter().all(|p| p.len() == t) && shares.len() == polys.len() * n);
    let limbs: Vec<i32> = polys.iter().flat_map(|p| pack_point_limbs(p)).collect();
    let sh = pack_scalars(shares);
    let mut verdict = vec![0u8; polys.len() * n];
    gpu.check(unsafe { sys::kb_dkg_verify_round_limbs(gpu.ctx, n, t, 0, polys.len(), limbs.as_ptr(), sh.as_ptr(), verdict.as_mut_ptr()) })?;
    Ok(verdict.into_iter().map(|v| v == 1).collect())
}

/// The flat (messages, offsets, signatures) of one keyed signature batch; a signature that is not 64 bytes long enters as
/// 64 zero bytes and its result is replaced by the reference's length error afterwards.
fn pack_keyed_batch(items: &[(&[u8], &[u8])]) -> (Vec<u8>, Vec<u64>, Vec<u8>) {
    let (mut msg, mut off, mut sig) = (vec![], vec![0u64], vec![]);
    for (m, s) in items {
        msg.extend_from_slice(m);
        off.push(msg.len() as u64);
        if s.len() == 64 {
            sig.extend_from_slice(s);
        } else {
            sig.extend_from_slice(&[0u8; 64]);
        }
    }
    (msg, off, sig)
}

/// `dkg_verify_round` plus the two Schnorr checks of the round (dkg.rs:531 on each deal, vss.rs:943 on each response) under
/// registered participant keys: `deals[d * n + i]` and `responses[d * n + i]` are (message, signature) of the deal dealer
/// `d` sent to verifier `i` and of that verifier's response, signed by key `d` of `dealers` and key `i` of `verifiers`.
/// `dealers` and `verifiers` may be the same key set (a new DKG) or two (resharing).  An empty `deals` or `responses`
/// skips that batch.  Returns (verdict, deal results, response results), each item what the scalar calls return.
pub fn dkg_process_round_keyed(gpu: &Gpu, dealers: &KeySet, verifiers: &KeySet, n: usize, polys: &[Vec<EdPoint>], shares: &[EdScalar],
                               deals: &[(&[u8], &[u8])], responses: &[(&[u8], &[u8])])
                               -> Result<(Vec<bool>, Vec<Result<(), SignatureError>>, Vec<Result<(), SignatureError>>), GpuError> {
    let t = polys.first().map(|p| p.len()).unwrap_or(0);
    let m = polys.len() * n;
    assert!(polys.iter().all(|p| p.len() == t) && shares.len() == m);
    assert!((deals.is_empty() || deals.len() == m) && (responses.is_empty() || responses.len() == m));
    let limbs: Vec<i32> = polys.iter().flat_map(|p| pack_point_limbs(p)).collect();
    let sh = pack_scalars(shares);
    let mut verdict = vec![0u8; m];
    let (dm, doff, dsig) = pack_keyed_batch(deals);
    let (rm, roff, rsig) = pack_keyed_batch(responses);
    let (mut dst, mut rst) = (vec![0u8; deals.len()], vec![0u8; responses.len()]);
    let sig_ptr = |items: &[(&[u8], &[u8])], s: &Vec<u8>| if items.is_empty() { std::ptr::null() } else { s.as_ptr() };
    gpu.check(unsafe {
        sys::kb_dkg_process_round_keyed(gpu.ctx, dealers.ks, verifiers.ks, n, t, 0, polys.len(), 1 /* KB_POINT_LIMBS40 */, limbs.as_ptr() as *const std::os::raw::c_void, sh.as_ptr(), verdict.as_mut_ptr(),
                                        dm.as_ptr(), doff.as_ptr(), sig_ptr(deals, &dsig), dst.as_mut_ptr(), rm.as_ptr(), roff.as_ptr(), sig_ptr(responses, &rsig), rst.as_mut_ptr())
    })?;
    let results = |items: &[(&[u8], &[u8])], st: Vec<u8>| -> Vec<Result<(), SignatureError>> {
        items.iter().zip(st).map(|((_, s), x)| status_to_result(if s.len() == 64 { x } else { 1 })).collect()
    };
    Ok((verdict.into_iter().map(|v| v == 1).collect(), results(deals, dst), results(responses, rst)))
}
