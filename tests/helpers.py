"""Shared test helpers: golden-file reader, C-oracle loader, deterministic input streams."""
import ctypes
import gzip
import hashlib
import os
import struct
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_sign_input():
    """tests/golden/sign_input.bin.gz -> list of (seed, pk, sig, msg); see make_golden.py."""
    raw = gzip.open(os.path.join(ROOT, "tests", "golden", "sign_input.bin.gz")).read()
    off, recs = 0, []
    while off < len(raw):
        seed, pk, sig = raw[off:off + 32], raw[off + 32:off + 64], raw[off + 64:off + 128]
        (ml,) = struct.unpack_from("<I", raw, off + 128)
        msg = raw[off + 132:off + 132 + ml]
        off += 132 + ml
        recs.append((seed, pk, sig, msg))
    assert len(recs) == 1024
    return recs


class COracle:
    """ctypes view of oracle/_build/liboracle.so (oracle/ref10_port.c)."""

    def __init__(self, path):
        L = ctypes.CDLL(path)
        self.L = L
        u8p = ctypes.c_char_p
        L.oracle_init.restype = None
        L.oracle_sha512.argtypes = [u8p, ctypes.c_size_t, u8p]
        L.oracle_sc_reduce64.argtypes = [u8p, u8p]
        L.oracle_sc_muladd.argtypes = [u8p, u8p, u8p, u8p]
        L.oracle_scalar_is_canonical.argtypes = [u8p]
        L.oracle_point_is_canonical.argtypes = [u8p]
        L.oracle_point_decode_ok.argtypes = [u8p]
        L.oracle_point_recode.argtypes = [u8p, u8p]
        L.oracle_point_has_small_order.argtypes = [u8p]
        L.oracle_mul_base.argtypes = [u8p, u8p]
        L.oracle_mul.argtypes = [u8p, u8p, u8p]
        L.oracle_point_add.argtypes = [u8p, u8p, u8p, ctypes.c_int]
        L.oracle_eddsa_verify.argtypes = [u8p, u8p, ctypes.c_size_t, u8p, ctypes.c_size_t]
        L.oracle_schnorr_verify.argtypes = [u8p, u8p, ctypes.c_size_t, u8p, ctypes.c_size_t]
        L.oracle_pubpoly_eval.argtypes = [u8p, u8p, ctypes.c_int, ctypes.c_uint32]
        L.oracle_vss_verify_deal.argtypes = [u8p, ctypes.c_int, ctypes.c_uint32, u8p]
        vp = ctypes.c_void_p
        L.oracle_mul_base_batch.argtypes = [ctypes.c_size_t, vp, vp, ctypes.c_int]
        L.oracle_mul_batch.argtypes = [ctypes.c_size_t, vp, vp, vp, ctypes.c_int]
        L.oracle_eddsa_verify_batch.argtypes = [ctypes.c_size_t, vp, vp, vp, vp, vp, ctypes.c_int]
        L.oracle_schnorr_verify_batch.argtypes = [ctypes.c_size_t, vp, vp, vp, vp, vp, ctypes.c_int]
        L.oracle_vss_verify_batch.argtypes = [vp, ctypes.c_int, ctypes.c_size_t, vp, vp, vp, ctypes.c_int]
        L.oracle_msm.argtypes = [u8p, ctypes.c_size_t, vp, vp]
        L.oracle_mul_base_limbs.argtypes = [vp, u8p]
        L.oracle_limbs_tobytes.argtypes = [u8p, vp]
        L.oracle_point_limbs.argtypes = [vp, u8p]
        L.oracle_sc_invert.argtypes = [u8p, u8p]
        L.oracle_rabin_verify_batch.argtypes = [vp, ctypes.c_int, u8p, ctypes.c_size_t, vp, vp, vp, vp, ctypes.c_int]
        L.oracle_dss_partial_batch.argtypes = [vp, vp, ctypes.c_int, u8p, ctypes.c_size_t, ctypes.c_size_t, vp, vp, vp, ctypes.c_int]
        L.oracle_dss_partial_check.argtypes = [u8p, u8p, ctypes.c_int, ctypes.c_uint32, u8p, ctypes.c_size_t, u8p, u8p]
        L.oracle_recover_commit.argtypes = [u8p, ctypes.c_int, vp, vp]
        L.oracle_recover_pub_poly.argtypes = [vp, ctypes.c_int, vp, vp]
        L.oracle_init()

    # ---- single-item wrappers
    def sha512(self, m):
        out = ctypes.create_string_buffer(64)
        self.L.oracle_sha512(m, len(m), out)
        return out.raw

    def sc_reduce64(self, d):
        out = ctypes.create_string_buffer(32)
        self.L.oracle_sc_reduce64(out, d)
        return out.raw

    def sc_muladd(self, a, b, c):
        out = ctypes.create_string_buffer(32)
        self.L.oracle_sc_muladd(out, a, b, c)
        return out.raw

    def scalar_is_canonical(self, s):
        return bool(self.L.oracle_scalar_is_canonical(s))

    def point_is_canonical(self, s):
        return bool(self.L.oracle_point_is_canonical(s))

    def point_decode_ok(self, s):
        return bool(self.L.oracle_point_decode_ok(s))

    def point_recode(self, s):
        out = ctypes.create_string_buffer(32)
        return out.raw if self.L.oracle_point_recode(out, s) else None

    def point_has_small_order(self, s):
        return self.L.oracle_point_has_small_order(s)

    def mul_base(self, a):
        out = ctypes.create_string_buffer(32)
        self.L.oracle_mul_base(out, a)
        return out.raw

    def mul(self, a, p):
        out = ctypes.create_string_buffer(32)
        return out.raw if self.L.oracle_mul(out, a, p) else None

    def point_add(self, p, q, subtract=False):
        out = ctypes.create_string_buffer(32)
        return out.raw if self.L.oracle_point_add(out, p, q, int(subtract)) else None

    def mul_base_limbs(self, a):
        out = np.empty(40, dtype=np.int32)
        self.L.oracle_mul_base_limbs(self._p(out), a)
        return out

    def point_limbs(self, enc):
        """40 int32 limbs (X, Y, Z, T) of a decodable encoding, as the reference holds it in memory."""
        out = np.empty(40, dtype=np.int32)
        assert self.L.oracle_point_limbs(self._p(out), bytes(enc)) == 1
        return out

    def limbs_tobytes(self, limbs):
        limbs = np.ascontiguousarray(limbs, dtype=np.int32)
        out = ctypes.create_string_buffer(32)
        self.L.oracle_limbs_tobytes(out, self._p(limbs))
        return out.raw

    def eddsa_verify(self, pk, msg, sig):
        return self.L.oracle_eddsa_verify(pk, msg, len(msg), sig, len(sig))

    def schnorr_verify(self, pk, msg, sig):
        return self.L.oracle_schnorr_verify(pk, msg, len(msg), sig, len(sig))

    def pubpoly_eval(self, commits, idx):
        out = ctypes.create_string_buffer(32)
        ok = self.L.oracle_pubpoly_eval(out, b"".join(commits), len(commits), idx)
        return out.raw if ok else None

    def vss_verify_deal(self, commits, idx, share):
        return self.L.oracle_vss_verify_deal(b"".join(commits), len(commits), idx, share)

    # ---- numpy batch wrappers (uint8 arrays, C-contiguous)
    @staticmethod
    def _p(a):
        return a.ctypes.data_as(ctypes.c_void_p)

    def mul_base_batch(self, scalars, nthreads=1):
        scalars = np.ascontiguousarray(scalars, dtype=np.uint8)
        out = np.empty_like(scalars)
        self.L.oracle_mul_base_batch(scalars.shape[0], self._p(scalars), self._p(out), nthreads)
        return out

    def mul_batch(self, scalars, points, nthreads=1):
        scalars = np.ascontiguousarray(scalars, dtype=np.uint8)
        points = np.ascontiguousarray(points, dtype=np.uint8)
        out = np.empty_like(scalars)
        self.L.oracle_mul_batch(scalars.shape[0], self._p(scalars), self._p(points), self._p(out), nthreads)
        return out

    def verify_batch(self, pk, msg, msg_off, sig, nthreads=1, schnorr=False):
        pk = np.ascontiguousarray(pk, dtype=np.uint8)
        sig = np.ascontiguousarray(sig, dtype=np.uint8)
        msg = np.ascontiguousarray(msg, dtype=np.uint8)
        msg_off = np.ascontiguousarray(msg_off, dtype=np.uint64)
        n = pk.shape[0]
        st = np.empty(n, dtype=np.uint8)
        fn = self.L.oracle_schnorr_verify_batch if schnorr else self.L.oracle_eddsa_verify_batch
        fn(n, self._p(pk), self._p(msg), self._p(msg_off), self._p(sig), self._p(st), nthreads)
        return st

    def vss_verify_batch(self, commits, idx, shares, nthreads=1):
        commits = np.ascontiguousarray(commits, dtype=np.uint8)
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        shares = np.ascontiguousarray(shares, dtype=np.uint8)
        out = np.empty(idx.shape[0], dtype=np.uint8)
        self.L.oracle_vss_verify_batch(self._p(commits), commits.shape[0], idx.shape[0], self._p(idx), self._p(shares), self._p(out), nthreads)
        return out

    def sc_invert(self, a):
        out = ctypes.create_string_buffer(32)
        self.L.oracle_sc_invert(out, a)
        return out.raw

    def rabin_verify_batch(self, commits, h_point, idx, f, g, nthreads=1):
        commits = np.ascontiguousarray(commits, dtype=np.uint8)
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        f, g = np.ascontiguousarray(f, dtype=np.uint8), np.ascontiguousarray(g, dtype=np.uint8)
        out = np.empty(idx.shape[0], dtype=np.uint8)
        self.L.oracle_rabin_verify_batch(self._p(commits), commits.shape[0], bytes(h_point), idx.shape[0], self._p(idx), self._p(f), self._p(g), self._p(out), nthreads)
        return out

    def dss_partial_batch(self, rand_commits, long_commits, msg, idx, partials, nthreads=1):
        r, l = np.ascontiguousarray(rand_commits, dtype=np.uint8), np.ascontiguousarray(long_commits, dtype=np.uint8)
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        p = np.ascontiguousarray(partials, dtype=np.uint8)
        out = np.empty(idx.shape[0], dtype=np.uint8)
        self.L.oracle_dss_partial_batch(self._p(r), self._p(l), r.shape[0], bytes(msg), len(msg), idx.shape[0], self._p(idx), self._p(p), self._p(out), nthreads)
        return out

    def dss_hash_sig(self, rand_commits, long_commits, msg):
        r, l = np.ascontiguousarray(rand_commits, dtype=np.uint8), np.ascontiguousarray(long_commits, dtype=np.uint8)
        h = ctypes.create_string_buffer(32)
        self.L.oracle_dss_partial_check(r.tobytes(), l.tobytes(), r.shape[0], 0, bytes(msg), len(msg), bytes(32), h)
        return h.raw

    def recover_commit(self, idx, points):
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        p = np.ascontiguousarray(points, dtype=np.uint8)
        out = ctypes.create_string_buffer(32)
        return out.raw if self.L.oracle_recover_commit(out, idx.shape[0], self._p(idx), self._p(p)) else None

    def recover_pub_poly(self, idx, points):
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        p = np.ascontiguousarray(points, dtype=np.uint8)
        out = np.empty((idx.shape[0], 32), dtype=np.uint8)
        return out if self.L.oracle_recover_pub_poly(self._p(out), idx.shape[0], self._p(idx), self._p(p)) else None

    def msm(self, scalars, points):
        scalars = np.ascontiguousarray(scalars, dtype=np.uint8)
        points = np.ascontiguousarray(points, dtype=np.uint8)
        out = ctypes.create_string_buffer(32)
        ok = self.L.oracle_msm(out, scalars.shape[0], self._p(scalars), self._p(points))
        return out.raw if ok else None


_ORACLE = None


def load_c_oracle():
    global _ORACLE
    if _ORACLE is None:
        path = os.path.join(ROOT, "oracle", "_build", "liboracle.so")
        src = os.path.join(ROOT, "oracle", "ref10_port.c")
        if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
        _ORACLE = COracle(path)
    return _ORACLE


L_ORDER = 2**252 + 27742317777372353535851937790883648493
P_FIELD = 2**255 - 19

# field elements (8 x 32-bit limbs, any value below 2^256) at the carry and wrap edges of the limb arithmetic
FE_EDGE = [0, 1, 2, 19, 38, P_FIELD - 1, P_FIELD, P_FIELD + 1, 2**255 - 1, 2**255, 2**255 + 18, 2**255 + 19, 2**256 - 1, 2**256 - 38, 2**256 - 39, 2**256 - 19,
           2**256 - 2**32, 2**224 - 1]


def half_step_special_inputs():
    """Challenges on which the lattice step sc_half (csrc/half.cuh) is hardest: rationals k/m of 8L (short vectors with
    tiny u, the Lehmer batches' awkward cases), powers of two and their small multiples, Fibonacci numbers (all
    quotients 1), and a few hand-picked values."""
    L = L_ORDER
    N = 8 * L
    special = [0, 1, 2, 3, 7, 8, L - 1, L - 2, L // 2, L // 3, 2**128, 2**127 + 1, 2**64, 2**200 + 5, (N // 3) % L, (N // 5 + 1) % L]
    for m in range(1, 400):
        for k in (1, 2, m // 2 + 1, m - 1):
            for d in (-2, -1, 0, 1, 2, 2**64, 2**128 + 1):
                special.append(((N * k) // m + d) % L)
    special += [(mul << e) % L for e in range(1, 253, 3) for mul in (1, 3, 5)]
    fa, fb = 1, 1
    while fb < L:
        special.append(fb)
        fa, fb = fb, fa + fb
    return special


def xof_bytes(seed: str, n: int) -> bytes:
    """Deterministic byte stream: BLAKE3-XOF of an ASCII seed — the construction behind the
    reference's suite.xof(Some(seed)) (suite.rs:128-133, xof/blake3/xof.rs:114-125).  Falls
    back to SHAKE-256 if the blake3 module is missing (only determinism matters here)."""
    try:
        import blake3

        return blake3.blake3(seed.encode()).digest(length=n)
    except ImportError:  # pragma: no cover
        return hashlib.shake_256(seed.encode()).digest(n)


def random_scalars(seed: str, n: int) -> np.ndarray:
    """n scalars < L as an (n,32) uint8 array (top 4 bits masked then reduced mod L;
    the distribution detail is irrelevant to parity)."""
    raw = np.frombuffer(xof_bytes(seed, 32 * n), dtype=np.uint8).reshape(n, 32).copy()
    out = np.empty_like(raw)
    for i in range(n):
        v = int.from_bytes(raw[i].tobytes(), "little") % L_ORDER
        out[i] = np.frombuffer(v.to_bytes(32, "little"), dtype=np.uint8)
    return out


# ---------------------------------------------------------------------------------------------
# adversarial signature batches (SURVEY §8d: valid items + every reject class the reference tests)
# ---------------------------------------------------------------------------------------------
WEAK_KEYS = [
    bytes(32),
    bytes([1]) + bytes(31),
    bytes.fromhex("26e8958fc2b227b045c3f489f2ef98f0d5dfac05d3c63339b13802886d53fc05"),
    bytes.fromhex("c7176a703d4dd84fba3c0b760d10670f2a2053fa2c39ccc64ec7fd7792ac037a"),
    bytes([0xEC]) + b"\xff" * 30 + b"\x7f",
]
NONCANONICAL = bytes([0xEF]) + b"\xff" * 31


def _off_curve(seed: int) -> bytes:
    """A canonical-looking 32-byte string that is not a curve point (found by search with the C oracle)."""
    C = load_c_oracle()
    k = 0
    while True:
        cand = hashlib.sha256(b"offcurve%d/%d" % (seed, k)).digest()
        cand = cand[:31] + bytes([cand[31] & 0x7F])
        if not C.point_decode_ok(cand):
            return cand
        k += 1


def mutate_signature(kind: int, rec, other):
    """Returns (pk, msg, sig) for mutation class `kind` of golden record `rec`."""
    seed, pk, sig, msg = rec
    L = L_ORDER
    s_plus_l = ((int.from_bytes(sig[32:], "little") + L) % (1 << 256)).to_bytes(32, "little")
    kind %= 24
    if kind == 0:
        return pk, msg, sig
    if kind == 1:
        m = bytearray(msg or b"\0"); m[0] ^= 1
        return pk, bytes(m), sig
    if kind == 2:
        return pk, msg, sig[:32] + s_plus_l
    if kind == 3:
        return pk, msg, NONCANONICAL + sig[32:]
    if kind == 4:
        return NONCANONICAL, msg, sig
    if kind in (5, 6, 7, 8, 9):
        return pk, msg, WEAK_KEYS[kind - 5] + sig[32:]
    if kind in (10, 11, 12, 13, 14):
        return WEAK_KEYS[kind - 10], msg, sig
    if kind == 15:
        return pk, msg, _off_curve(1) + sig[32:]
    if kind == 16:
        return _off_curve(2), msg, sig
    if kind == 17:   # quirk range (SURVEY §A1): canonical y reported non-canonical
        return pk, msg, bytes([0x14 + (len(msg) % 0xD9)]) + b"\xff" * 30 + b"\x7f" + sig[32:]
    if kind == 18:
        return bytes([0x14 + (len(msg) % 0xD9)]) + b"\xff" * 30 + b"\xff", msg, sig
    if kind == 19:   # several things wrong at once: the verifiers' check ORDER decides
        return NONCANONICAL, msg, NONCANONICAL + s_plus_l
    if kind == 20:
        return NONCANONICAL, msg, _off_curve(3) + sig[32:]
    if kind == 21:
        return _off_curve(4), msg, WEAK_KEYS[3] + s_plus_l
    if kind == 22:   # a different (valid) R
        return pk, msg, other[2][:32] + sig[32:]
    w = bytearray(WEAK_KEYS[1]); w[31] |= 0x80   # identity with the sign bit set (x = 0, SURVEY §A2)
    return pk, msg, bytes(w) + sig[32:]


def make_sig_batch(records, n: int, bad_every: int = 4):
    """n (pk, msg, sig) triples cycling through the golden records; every `bad_every`-th item is a
    mutation, cycling through all classes.  Returns (pks, msgs, sigs) lists."""
    pks, msgs, sigs = [], [], []
    kind = 1
    for i in range(n):
        rec = records[i % len(records)]
        if bad_every and i % bad_every == bad_every - 1:
            pk, msg, sig = mutate_signature(kind, rec, records[(i + 7) % len(records)])
            kind += 1
        else:
            _, pk, sig, msg = rec
        pks.append(pk); msgs.append(msg); sigs.append(sig)
    return pks, msgs, sigs


def pack_batch(pks, msgs, sigs):
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64)
    flat = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy()
    pk = np.frombuffer(b"".join(pks), dtype=np.uint8).reshape(-1, 32).copy()
    sg = np.frombuffer(b"".join(sigs), dtype=np.uint8).reshape(-1, 64).copy()
    return pk, flat, off, sg


def make_mixed_order_sigs(count: int, seed: int = 1):
    """Signatures whose public key AND R carry a small-order component (both pass the reference's small-order
    filter, which only rejects points that are ENTIRELY of small order).  With A = a*B + T, R = r*B + T' the
    reference's cofactorless equation s*B == R + h*A holds iff T' + h*T == 0.  Returns `count` triples
    (pk, msg, sig) for which it holds ("accept") and `count` near misses for which it fails ("reject") although
    8*(s*B - R - h*A) == 0 — the inputs on which a cofactored, a batched or a mod-L-shortened verifier would
    disagree with the reference."""
    import random

    from oracle import ed25519_bigint as O

    rnd = random.Random(seed)
    tors = [O.point_decode(k) for k in O.WEAK_KEYS[2:4]]          # the two encodings of order-8 points
    t8 = tors[0]
    torsion = [O.IDENTITY]
    for _ in range(7):
        torsion.append(O.point_add(torsion[-1], t8))
    good, bad = [], []
    while len(good) < count or len(bad) < count:
        a = rnd.randrange(1, O.L)
        r = rnd.randrange(1, O.L)
        T = torsion[rnd.randrange(1, 8)]
        Tp = torsion[rnd.randrange(0, 8)]
        A = O.point_add(O._mul_int(a, O.BASE), T)
        R = O.point_add(O._mul_int(r, O.BASE), Tp)
        pk, rb = O.point_encode(A), O.point_encode(R)
        msg = rnd.randbytes(rnd.randrange(0, 100))
        h = int.from_bytes(O.challenge(rb, pk, msg), "little")
        s = (r + h * a) % O.L
        sig = rb + s.to_bytes(32, "little")
        holds = O.point_eq(O.point_add(Tp, O._mul_int(h, T)), O.IDENTITY)
        (good if holds else bad).append((pk, msg, sig))
    return good[:count], bad[:count]
