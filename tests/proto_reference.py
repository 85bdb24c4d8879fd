"""Exact references for the protocol entry points: interpolation in the exponent (recover_commit, recover_pub_poly,
resharing_key), polynomial evaluation (PubPoly / PriPoly, VSS share checks), the DSS challenge and session ids.

Every one of them has an answer that plain Python integers give exactly: the device result is (exact scalar) * B,
and the scalar is a Horner evaluation, a Lagrange-weighted sum or a hash, mod L.  The evaluation point of index i is
x = i + 1, an integer up to 2^32 that the kernels hold in two 32-bit words (and as a NAF of up to 33 digits).
`index_set` gives the 32-bit indices at which that arithmetic carries, wraps or runs longest.

Needs no GPU.  tests/test_proto_reference_cpu.py holds these helpers to oracle/ed25519_bigint.py at small sizes;
tests/test_gpu_proto_shapes.py holds the device to them at the DKG shape.
"""
import hashlib

import numpy as np

from oracle import ed25519_bigint as O

L = O.L

# Indices (x = i + 1) in the order index_set takes them:
#   2^32 - 1, 2^31 - 1, 2^31, 2^32 - 2   x = 2^32 (the upper word of x, a 33-digit NAF), 2^31, 2^31 + 1, 2^32 - 1
#                                        (33-digit NAF 1 0 .. 0 -1); 2^31 - 1 / 2^32 - 1 and 0 / 2^31 lie 2^31 apart
#   0, 1, 2                              the smallest nodes, adjacent
#   0xAAAAAAAA                           x = 0xAAAAAAAB: 33 NAF digits, 17 of them non-zero (the densest a 33-digit NAF gets)
#   0x55555555                           x = 0x55555556: 32 digits, 16 non-zero
#   0xAAAAAAA9, 0x55555554               x = 0xAAAAAAAA, 0x55555555 (31 digits, 16 non-zero); each adjacent to the one above
#   0x2AAAAAAA, 0xD5555555               2^31 below 0xAAAAAAAA and 2^31 above 0x55555555
SPECIAL = [2**32 - 1, 2**31 - 1, 2**31, 2**32 - 2, 0, 1, 2, 0xAAAAAAAA, 0x55555555, 0xAAAAAAA9, 0x55555554, 0x2AAAAAAA, 0xD5555555]


def naf(x: int):
    """Non-adjacent form of x >= 1, least significant digit first: the digits kb_naf_from (csrc/poly.cuh) computes."""
    d = []
    while x:
        z = 0
        if x & 1:
            z = 2 - (x & 3)
            x -= z
        d.append(z)
        x >>= 1
    return d


def index_set(k: int, seed: int = 0) -> np.ndarray:
    """k distinct 32-bit indices, unsorted: the first min(k, len(SPECIAL)) of SPECIAL, then seeded uniform 32-bit
    values; the whole set in a seeded random order."""
    rng = np.random.default_rng([seed, 0x1D])
    out = list(SPECIAL[:k])
    have = set(out)
    while len(out) < k:
        for v in rng.integers(0, 2**32, size=k, dtype=np.uint64).tolist():
            if v not in have and len(out) < k:
                have.add(v)
                out.append(v)
    return np.array(out, dtype=np.uint32)[rng.permutation(k)]


def small_index_set(k: int, n: int, seed: int = 0) -> np.ndarray:
    """k distinct indices below n, unsorted (a realistic set of qualified nodes)."""
    return np.random.default_rng([seed, 0x5E]).choice(n, size=k, replace=False).astype(np.uint32)


# ---- scalars as Python integers and as (n, 32) little-endian bytes ------------------------------------------------
def to_bytes(vals) -> np.ndarray:
    return np.frombuffer(b"".join((int(v) % 2**256).to_bytes(32, "little") for v in vals), dtype=np.uint8).reshape(-1, 32).copy()


def to_ints(a):
    """(n, 32) uint8 -> list of n Python ints."""
    w = np.ascontiguousarray(a, dtype=np.uint8).reshape(-1, 32).view("<u8").astype(object)
    return (w[:, 0] | (w[:, 1] << 64) | (w[:, 2] << 128) | (w[:, 3] << 192)).tolist()


def scalars(n: int, seed: int) -> list:
    """n random scalars below L (252 random bits; L - 1, L - 2, 1 and 0 at the first four positions when n >= 16)."""
    b = np.random.default_rng([seed, 0x5C]).integers(0, 256, size=(n, 32), dtype=np.uint8)
    b[:, 31] &= 0x0F
    v = to_ints(b)
    if n >= 16:
        v[:4] = [L - 1, L - 2, 1, 0]
    return v


# ---- the operations --------------------------------------------------------------------------------------------------
def poly_eval(coeffs, x: int) -> int:
    """sum_c coeffs[c] * x^c mod L by Horner's rule (PriPoly::eval at index x - 1; PubPoly::eval's discrete log)."""
    v = 0
    for c in reversed(coeffs):
        v = (v * x + c) % L
    return v


def poly_eval_many(coeffs, xs) -> list:
    """poly_eval at every x of xs, Horner steps vectorised over the points."""
    xa = np.array([int(x) for x in xs], dtype=object)
    v = np.zeros(len(xa), dtype=object)
    for c in reversed(coeffs):
        v = (v * xa + c) % L
    return v.tolist()


def lagrange_at_zero(xs) -> list:
    """lam_i = prod_{j != i} x_j / prod_{j != i} (x_j - x_i) mod L: the weights of recover_commit (share/poly.rs:583-597),
    so that sum_i lam_i p(x_i) = p(0) for every polynomial p of degree below len(xs).  The nodes must be distinct."""
    xs = [int(x) for x in xs]
    xa = np.array(xs, dtype=object)
    den = np.ones(len(xs), dtype=object)
    for j, xj in enumerate(xs):
        d = xj - xa
        d[j] = 1
        den = den * d % L
    num = 1
    for x in xs:
        num = num * x % L
    return [num * pow(x * int(dn) % L, -1, L) % L for x, dn in zip(xs, den)]


def weighted_sum(weights, vals) -> int:
    return sum(w * v for w, v in zip(weights, vals)) % L


def challenge(r32: bytes, a32: bytes, msg: bytes) -> int:
    """SHA-512(R || A || msg) mod L (hash_sig, sign/dss/dss_sig.rs:312-326)."""
    return int.from_bytes(hashlib.sha512(bytes(r32) + bytes(a32) + bytes(msg)).digest(), "little") % L


def session_id(dealer32: bytes, verifiers32, commits32, t: int) -> bytes:
    """SHA-256(dealer || verifiers || commits || t as u32 LE) over canonical encodings (vss/pedersen/vss.rs:1069-1090)."""
    h = hashlib.sha256(bytes(dealer32))
    h.update(np.ascontiguousarray(verifiers32, dtype=np.uint8).tobytes())
    h.update(np.ascontiguousarray(commits32, dtype=np.uint8).tobytes())
    h.update(int(t).to_bytes(4, "little"))
    return h.digest()
