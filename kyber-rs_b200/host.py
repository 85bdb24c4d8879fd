"""Host-side mirror of the reference's operator surface for the edwards25519 hot path.

Same names, argument meaning and error behaviour as kyber-rs (paths relative to
/root/reference/src), with batch entry points added next to each scalar one:

    group::Point / edwards25519::Point   (group.rs:85, group/edwards25519/point.rs)   -> Point
    group::Scalar / edwards25519::Scalar (group.rs:22, group/edwards25519/scalar.rs)  -> Scalar
    share::poly::PubPoly                 (share/poly.rs:398)                          -> PubPoly
    sign::eddsa::verify[_with_checks]    (sign/eddsa/eddsa_sig.rs:159-219)            -> eddsa_verify*
    sign::schnorr::verify                (sign/schnorr/schnorr_sig.rs:53-126)         -> schnorr_verify*
    vss::pedersen Aggregator::verify_deal group math (share/vss/pedersen/vss.rs:899)  -> vss_verify_deal*
    SignatureError / MarshallingError    (sign/error.rs, encoding/encodings.rs:30)    -> same names

ALL arithmetic goes through the C ABI (``binding.Context``) and therefore runs on the GPU; this
module holds no field, curve or scalar arithmetic of its own and fails loudly without a GPU.
"""
from __future__ import annotations

import numpy as np

from .binding import Context, SIG_STATUS_NAMES, pack_messages

_CTX = None


def default_context() -> Context:
    global _CTX
    if _CTX is None:
        _CTX = Context(0)
    return _CTX


def set_default_context(ctx: Context):
    global _CTX
    _CTX = ctx


class MarshallingError(ValueError):
    """encoding::MarshallingError::InvalidInput (encoding/encodings.rs:30-39)."""


class SignatureError(Exception):
    """sign::error::SignatureError; str() is the reference's #[error("...")] text."""

    def __init__(self, status: int):
        self.status = int(status)
        super().__init__(SIG_STATUS_NAMES[self.status])


_ONE = (1).to_bytes(32, "little")
_ZERO = bytes(32)
_L_MINUS_1 = bytes.fromhex("ecd3f55c1a631258d69cf7a2def9de1400000000000000000000000000000010")   # scalar_test.rs:38-46
_BASE = bytes.fromhex("58" + "66" * 31)  # compress(B): y = 4/5, x positive (constants.rs:70 BASEEXT)
_NULL = _ONE                              # compress((0,1))


class Scalar:
    """edwards25519::Scalar — 32 little-endian bytes, NOT necessarily reduced (scalar.rs:24, SURVEY §A3)."""

    __slots__ = ("v",)

    def __init__(self, v: bytes = _ZERO):
        assert len(v) == 32
        self.v = bytes(v)

    # Scalar::set_bytes (scalar.rs:175): little-endian integer of any length <= 64 bytes, mod L
    @staticmethod
    def set_bytes(b: bytes, ctx: Context | None = None) -> "Scalar":
        assert len(b) <= 64
        d = np.frombuffer(b.ljust(64, b"\0"), dtype=np.uint8)
        return Scalar((ctx or default_context()).sc_reduce64_batch(d)[0].tobytes())

    # Scalar::set_int64 (scalar.rs:152) for non-negative values
    @staticmethod
    def set_int64(v: int) -> "Scalar":
        assert 0 <= v < 2**63
        return Scalar(v.to_bytes(32, "little"))

    @staticmethod
    def one() -> "Scalar":
        return Scalar(_ONE)

    @staticmethod
    def zero() -> "Scalar":
        return Scalar(_ZERO)

    # BinaryUnmarshaler (scalar.rs:102-112): raw copy, no reduction
    @staticmethod
    def unmarshal_binary(data: bytes) -> "Scalar":
        if len(data) != 32:
            raise MarshallingError("wrong size buffer")
        return Scalar(data)

    # BinaryMarshaler (scalar.rs:91-100): reduces mod L
    def marshal_binary(self) -> bytes:
        return Scalar.set_bytes(self.v).v

    def _muladd(self, b: "Scalar", c: "Scalar") -> "Scalar":
        out = default_context().sc_muladd_batch(np.frombuffer(self.v, np.uint8), np.frombuffer(b.v, np.uint8), np.frombuffer(c.v, np.uint8))
        return Scalar(out[0].tobytes())

    def __mul__(self, o: "Scalar") -> "Scalar":   # scalar.rs:132 (sc_mul)
        return self._muladd(o, Scalar(_ZERO))

    def __add__(self, o: "Scalar") -> "Scalar":   # scalar.rs:138 (sc_add)
        return self._muladd(Scalar(_ONE), o)

    def sub(self, a: "Scalar", b: "Scalar") -> "Scalar":     # scalar.rs:162 (sc_sub): a - b = a + (L-1)*b
        return b._muladd(Scalar(_L_MINUS_1), a)

    def neg(self, a: "Scalar") -> "Scalar":                  # scalar.rs:216
        return a._muladd(Scalar(_L_MINUS_1), Scalar(_ZERO))

    def inv(self, a: "Scalar") -> "Scalar":                  # scalar.rs:192-214: a^(L-2)
        return Scalar(default_context().sc_invert_batch(np.frombuffer(a.v, np.uint8))[0].tobytes())

    def div(self, a: "Scalar", b: "Scalar") -> "Scalar":     # scalar.rs:185
        return a * Scalar().inv(b)

    def __eq__(self, o) -> bool:                  # scalar.rs:78: raw bytes
        return isinstance(o, Scalar) and self.v == o.v

    def __hash__(self):
        return hash(self.v)

    # ScalarCanCheckCanonical::is_canonical (scalar.rs:54): answered by the verifier kernels' own
    # check — a signature whose s is non-canonical is reported as SignatureNotCanonical.
    def __repr__(self):
        return f"Ed25519Scalar({self.v.hex()})"


class Point:
    """edwards25519::Point held as its canonical 32-byte encoding (what Point::eq compares,
    point.rs:227-241)."""

    __slots__ = ("b",)

    def __init__(self, b: bytes = _NULL):
        assert len(b) == 32
        self.b = bytes(b)

    @staticmethod
    def null() -> "Point":                         # point.rs:79
        return Point(_NULL)

    @staticmethod
    def base() -> "Point":                         # point.rs:85
        return Point(_BASE)

    # BinaryUnmarshaler (point.rs:43-51): error text as in the reference
    @staticmethod
    def unmarshal_binary(data: bytes, ctx: Context | None = None) -> "Point":
        if len(data) != 32:
            raise MarshallingError("invalid Ed25519 curve point")
        out, st = (ctx or default_context()).point_recode_batch(np.frombuffer(data, np.uint8))
        if st[0]:
            raise MarshallingError("invalid Ed25519 curve point")
        return Point(out[0].tobytes())

    def marshal_binary(self) -> bytes:             # point.rs:35-41
        return self.b

    # Point::mul (point.rs:207-225): p=None means the standard base
    def mul(self, s: Scalar, p: "Point | None" = None) -> "Point":
        ctx = default_context()
        sv = np.frombuffer(s.v, np.uint8)
        if p is None:
            return Point(ctx.point_mul_base_batch(sv)[0].tobytes())
        out, st = ctx.point_mul_batch(sv, np.frombuffer(p.b, np.uint8))
        assert not st[0]
        return Point(out[0].tobytes())

    def add(self, a: "Point", b: "Point") -> "Point":   # point.rs:179
        out, st = default_context().point_add_batch(np.frombuffer(a.b, np.uint8), np.frombuffer(b.b, np.uint8))
        assert not st[0]
        return Point(out[0].tobytes())

    def sub(self, a: "Point", b: "Point") -> "Point":   # point.rs:190
        out, st = default_context().point_add_batch(np.frombuffer(a.b, np.uint8), np.frombuffer(b.b, np.uint8), subtract=True)
        assert not st[0]
        return Point(out[0].tobytes())

    def neg(self, a: "Point") -> "Point":               # point.rs:201
        return self.sub(Point.null(), a)

    def __eq__(self, o) -> bool:                        # point.rs:227
        return isinstance(o, Point) and self.b == o.b

    def __hash__(self):
        return hash(self.b)

    # PointCanCheckCanonicalAndSmallOrder (point.rs:286, :322)
    @staticmethod
    def is_canonical(b: bytes) -> bool:
        if len(b) != 32:
            return False
        return bool(default_context().point_check_batch(np.frombuffer(b, np.uint8))[0] & 1)

    def has_small_order(self) -> bool:
        return bool(default_context().point_check_batch(np.frombuffer(self.b, np.uint8))[0] & 2)

    # ---- batch entry points behind the same trait ------------------------------------------
    @staticmethod
    def mul_batch(scalars, points=None, flags=0, ctx: Context | None = None):
        """scalars: (n,32) uint8; points: None (base point), (1,32) shared or (n,32)."""
        ctx = ctx or default_context()
        if points is None:
            return ctx.point_mul_base_batch(scalars, flags)
        return ctx.point_mul_batch(scalars, points, flags)

    def __repr__(self):
        return f"Ed25519Point({self.b.hex()})"


class PubPoly:
    """share::poly::PubPoly over the standard base (share/poly.rs:398)."""

    def __init__(self, commits):
        self.commits = [c if isinstance(c, Point) else Point(c) for c in commits]

    def threshold(self) -> int:
        return len(self.commits)

    def _flat(self):
        return np.frombuffer(b"".join(c.b for c in self.commits), np.uint8)

    def eval(self, i: int) -> Point:                    # poly.rs:457-469
        return self.eval_batch([i])[0]

    def eval_batch(self, idx, ctx: Context | None = None):
        idx = np.asarray(idx, dtype=np.uint32)
        out, st = (ctx or default_context()).pubpoly_eval_batch(self._flat(), self.threshold(), np.zeros_like(idx), idx)
        assert not st.any()
        return [Point(o.tobytes()) for o in out]

    def check(self, i: int, share: Scalar) -> bool:     # poly.rs:526-530
        return bool(self.check_batch([i], [share])[0])

    def check_batch(self, idx, shares, ctx: Context | None = None):
        idx = np.asarray(idx, dtype=np.uint32)
        sh = np.frombuffer(b"".join(s.v if isinstance(s, Scalar) else bytes(s) for s in shares), np.uint8)
        return (ctx or default_context()).vss_verify_deals_batch(self._flat(), self.threshold(), np.zeros_like(idx), idx, sh)

    def add(self, q: "PubPoly") -> "PubPoly":           # poly.rs:486-509
        if self.threshold() != q.threshold():
            raise ValueError("different number of coefficients")
        out, st = default_context().point_add_batch(self._flat(), q._flat())
        assert not st.any()
        return PubPoly([Point(o.tobytes()) for o in out])

    def equal(self, q: "PubPoly") -> bool:              # poly.rs:511-523
        return [c.b for c in self.commits] == [c.b for c in q.commits]


# ---- signatures -------------------------------------------------------------------------------
def _verify_batch(pks, msgs, sigs, schnorr, ctx):
    ctx = ctx or default_context()
    n = len(pks)
    assert len(msgs) == n and len(sigs) == n
    status = np.zeros(n, dtype=np.uint8)
    if any(len(pk) != 32 for pk in pks):
        raise ValueError("public keys must be 32-byte encodings (eddsa::verify marshals a Point, eddsa_sig.rs:216-219)")
    good = [k for k in range(n) if len(sigs[k]) == 64]
    for k in range(n):
        if len(sigs[k]) != 64:
            status[k] = 1    # InvalidSignatureLength (eddsa_sig.rs:161, schnorr_sig.rs:68)
    if good:
        flat, off = pack_messages([msgs[k] for k in good])
        pk = np.frombuffer(b"".join(pks[k] for k in good), np.uint8)
        sg = np.frombuffer(b"".join(sigs[k] for k in good), np.uint8)
        status[good] = ctx.verify_batch(pk, flat, off, sg, schnorr=schnorr)
    return status


def eddsa_verify_batch(pks, msgs, sigs, ctx: Context | None = None):
    """eddsa::verify_with_checks for n (public key bytes, message, signature) triples -> status[n]."""
    return _verify_batch(pks, msgs, sigs, False, ctx)


def schnorr_verify_batch(pks, msgs, sigs, ctx: Context | None = None):
    return _verify_batch(pks, msgs, sigs, True, ctx)


def eddsa_verify_with_checks(public_key: bytes, msg: bytes, sig: bytes):
    """sign/eddsa/eddsa_sig.rs:159 — returns None or raises SignatureError."""
    st = int(eddsa_verify_batch([public_key], [msg], [sig])[0])
    if st:
        raise SignatureError(st)


def eddsa_verify(public: Point, msg: bytes, sig: bytes):
    """sign/eddsa/eddsa_sig.rs:216."""
    eddsa_verify_with_checks(public.marshal_binary(), msg, sig)


def schnorr_verify(public: Point, msg: bytes, sig: bytes):
    """sign/schnorr/schnorr_sig.rs:114."""
    st = int(schnorr_verify_batch([public.marshal_binary()], [msg], [sig])[0])
    if st:
        raise SignatureError(st)


def eddsa_sign_batch(seeds, msgs, ctx: Context | None = None):
    """EdDSA::sign (sign/eddsa/eddsa_sig.rs:120-152) for n (32-byte seed, message) pairs -> (sigs[n,64], pks[n,32])."""
    flat, off = pack_messages(list(msgs))
    return (ctx or default_context()).eddsa_sign_batch(np.frombuffer(b"".join(seeds), np.uint8), flat, off)


# ---- VSS / DKG / MSM --------------------------------------------------------------------------
def vss_verify_deal(commits, i: int, share: Scalar) -> bool:
    """Group math of Aggregator::verify_deal (share/vss/pedersen/vss.rs:899-912)."""
    return PubPoly(commits).check(i, share)


def msm(scalars, points, ctx: Context | None = None) -> Point:
    """sum_i Point::mul(s_i, P_i) folded with Point::add."""
    enc, bad = (ctx or default_context()).msm(scalars, points)
    if bad:
        raise MarshallingError("invalid Ed25519 curve point")
    return Point(enc)


def vss_rabin_verify_deals_batch(commits, idx, f_shares, g_shares, h_point: Point, ctx: Context | None = None):
    """vss::rabin verify_deal group math (share/vss/rabin/vss.rs:889-900): fi*G + gi*H == eval(fi.i) on
    canonical encodings, for m (index, f share, g share) triples against one polynomial — one C-ABI call
    (kb_vss_rabin_verify_deals_batch): evaluation, both constant-time multiplications and the comparison stay on the device."""
    ctx = ctx or default_context()
    poly = PubPoly(commits)
    idx = np.asarray(idx, dtype=np.uint32)
    f = np.frombuffer(b"".join(s.v if isinstance(s, Scalar) else bytes(s) for s in f_shares), np.uint8).reshape(-1, 32)
    g = np.frombuffer(b"".join(s.v if isinstance(s, Scalar) else bytes(s) for s in g_shares), np.uint8).reshape(-1, 32)
    return ctx.vss_rabin_verify_deals_batch(poly._flat(), poly.threshold(), np.frombuffer(h_point.b, np.uint8), np.zeros_like(idx), idx, f, g)


def dss_verify_partials_batch(random_commits, long_commits, idx, partials, msg: bytes, ctx: Context | None = None):
    """Group math of DSS::process_partial_sig (sign/dss/dss_sig.rs:263-273) for m partial signatures of one session:
    partial_i * B == random_poly.eval(i) + hash_sig() * long_poly.eval(i), hash_sig = H(R || A || msg) (:312-326).
    One C-ABI call (kb_dss_verify_partials).  Returns (verdict[m], hash Scalar)."""
    ctx = ctx or default_context()
    rp, lp = PubPoly(random_commits), PubPoly(long_commits)
    p = np.frombuffer(b"".join(s.v if isinstance(s, Scalar) else bytes(s) for s in partials), np.uint8).reshape(-1, 32)
    verdict, h = ctx.dss_verify_partials(rp._flat(), lp._flat(), msg, np.asarray(idx, dtype=np.uint32), p)
    return verdict, Scalar(h)


def session_id(dealer: Point, verifiers, commitments, t: int, ctx: Context | None = None) -> bytes:
    """session_id (share/vss/pedersen/vss.rs:1069-1090)."""
    ctx = ctx or default_context()
    flat = lambda pts: np.frombuffer(b"".join(p.b for p in pts), np.uint8)
    out, st = ctx.vss_session_ids(np.frombuffer(dealer.b, np.uint8), flat(verifiers), flat(commitments), t)
    if st[0]:
        raise MarshallingError("invalid Ed25519 curve point")
    return out[0].tobytes()


def find_pub(points, to_find: Point, ctx: Context | None = None):
    """find_pub (share/dkg/pedersen/dkg.rs:1109-1116): (index, found)."""
    i = int((ctx or default_context()).find_pub_batch(np.frombuffer(b"".join(p.b for p in points), np.uint8), np.frombuffer(to_find.b, np.uint8))[0])
    return (i, True) if i >= 0 else (0, False)


def schnorr_sign_batch(privates, msgs, nonces, ctx: Context | None = None):
    """schnorr::sign (sign/schnorr/schnorr_sig.rs:25-47) for n (private scalar, message) pairs with the
    nonces k supplied by the caller (the reference draws them from its RNG): R = k*B, h = H(R || A || M),
    s = k + x*h.  Returns (signatures[n,64], public keys[n,32]).  One C-ABI call (kb_schnorr_sign_batch): both
    fixed-base multiplications run constant-time, and the secrets and nonces are wiped from device scratch."""
    ctx = ctx or default_context()
    x = np.frombuffer(b"".join(s.v if isinstance(s, Scalar) else bytes(s) for s in privates), np.uint8).reshape(-1, 32)
    k = np.frombuffer(b"".join(s.v if isinstance(s, Scalar) else bytes(s) for s in nonces), np.uint8).reshape(-1, 32)
    flat, off = pack_messages(list(msgs))
    return ctx.schnorr_sign_batch(x, k, flat, off)


def _xy_commit(shares, t: int):
    """xy_commit (share/poly.rs:535-562): the first t present shares in index order."""
    good = sorted(((i, p) for i, p in shares if p is not None), key=lambda s: s[0])[:t]
    if len(good) < t:
        raise ValueError("not enough good public shares to reconstruct secret commitment")   # PolyError::NotEnoughtGoodPublics
    return good


def recover_commit(shares, t: int, n: int, ctx: Context | None = None) -> Point:
    """share::poly::recover_commit (share/poly.rs:566-603): Lagrange interpolation in the exponent of the
    secret commitment p(0) from public shares [(index, Point), ...].  One C-ABI call (kb_recover_commit_batch):
    the Lagrange coefficients, the t scalar multiplications and their sum are computed on the device."""
    good = _xy_commit(shares, t)
    out, st = (ctx or default_context()).recover_commit_batch([i for i, _ in good], np.frombuffer(b"".join(p.b for _, p in good), np.uint8))
    if st[0]:
        raise MarshallingError("invalid Ed25519 curve point")
    return Point(out[0].tobytes())


def recover_pub_poly(shares, t: int, n: int, ctx: Context | None = None) -> PubPoly:
    """share::poly::recover_pub_poly (share/poly.rs:607-635)."""
    good = _xy_commit(shares, t)
    out, st = (ctx or default_context()).recover_pub_poly([i for i, _ in good], np.frombuffer(b"".join(p.b for _, p in good), np.uint8))
    if st.any():
        raise MarshallingError("invalid Ed25519 curve point")
    return PubPoly([Point(o.tobytes()) for o in out])


def resharing_key_commits(deal_commits, old_t: int, new_t: int, share_index: int, share: Scalar, ctx: Context | None = None):
    """The group math of resharing_key (share/dkg/pedersen/dkg.rs:996-1031): deal_commits = {old node index: [new_t
    Points]} of the qualified deals; returns the new_t commitments of the new public polynomial and whether it checks
    against the new private share (DKGError::ShareDoesNotMatchPublicPoly otherwise)."""
    good = sorted(deal_commits.items())[:old_t]
    if len(good) < old_t:
        raise ValueError("not enough good public shares to reconstruct secret commitment")
    flat = np.frombuffer(b"".join(p.b for _, row in good for p in row[:new_t]), np.uint8)
    out, st, chk = (ctx or default_context()).dkg_resharing_key(new_t, [i for i, _ in good], flat, share_index, np.frombuffer(share.v, np.uint8))
    if st.any():
        raise MarshallingError("invalid Ed25519 curve point")
    return [Point(o.tobytes()) for o in out], chk
