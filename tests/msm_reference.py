"""Exact closed-form reference for multi-scalar multiplication at any size.

The points have known discrete logs: P_i = r_i*B + t_i*T8, with B the base point, T8 a point of order 8 and
t_i in 0..7.  For any raw 32-byte scalars s_i,

    sum_i Point::mul(s_i, P_i) = (sum_i eff(s_i) * r_i mod L) * B + (sum_i s_i * t_i mod 8) * T8

where eff(s) is the integer the reference's scalar multiplication actually multiplies by (SURVEY §A3,
`O.scalar_effective`, `sc_effective` in csrc/sc.cuh), and eff(s) = s (mod 8) in every case.  The right-hand side
costs two scalar products, one point multiplication and one point addition, so an MSM of 2^24 points is checked
without any curve arithmetic per point.  The scalar products are exact: 16-bit limbs, multiplied as float64
matrices over blocks of 2^18 rows, so that no partial sum reaches 2^53.

Needs no GPU.  `gpu_points` builds the points with a context's scalar-multiplication kernels; `oracle_points`
builds them with the C oracle on the host.
"""
import numpy as np

from oracle import ed25519_bigint as O

L = O.L
T8 = O.WEAK_KEYS[2]                       # encoding of a point of order 8
_T8_PT = O.point_decode(T8)
TORSION = np.frombuffer(b"".join(O.point_encode(O._mul_int(t, _T8_PT)) for t in range(8)), dtype=np.uint8).reshape(8, 32).copy()
_C8 = sum(8 << (4 * i) for i in range(63))
CARRY_EDGE = 2**252 - _C8                 # low 252 bits >= CARRY_EDGE <=> the radix-16 recoding carries into nibble 63
_BLOCK = 1 << 18                          # rows per float64 product: 2^18 * 2^32 < 2^53


def to_bytes(vals):
    """Python ints (mod 2^256) -> (n, 32) uint8."""
    return np.frombuffer(b"".join((v % 2**256).to_bytes(32, "little") for v in vals), dtype=np.uint8).reshape(-1, 32).copy()


def to_ints(a):
    return [int.from_bytes(bytes(r), "little") for r in np.asarray(a, dtype=np.uint8).reshape(-1, 32)]


def _limbs(a):
    """(n, 32) uint8 -> (16, n) int64: row j holds 16-bit limb j of every scalar."""
    return np.ascontiguousarray(np.ascontiguousarray(a, dtype=np.uint8).view("<u2").T, dtype=np.int64)


def _const_limbs(v):
    return _limbs(np.frombuffer(v.to_bytes(32, "little"), dtype=np.uint8).reshape(1, 32))


def _at_least(words, v):
    """words >= v for (n, 4) little-endian uint64 words and an int v, vectorised."""
    res = np.zeros(words.shape[0], dtype=bool)
    eq = np.ones(words.shape[0], dtype=bool)
    for j in (3, 2, 1, 0):
        vj = np.uint64((v >> (64 * j)) & (2**64 - 1))
        res |= eq & (words[:, j] > vj)
        eq &= words[:, j] == vj
    return res | eq


def effective(scalars):
    """The effective scalars of raw 32-byte scalars, vectorised, as eff = mag - 2^252 * neg with mag >= 0:
    (mag limbs (16, n) int64, neg (n,) bool).  The low 252 bits and the carry of the radix-16 recoding decide:
    top nibble + carry <= 8 -> s itself; otherwise the top digit is dropped, leaving low252 without a carry and
    low252 - 2^252 (negative) with one."""
    scalars = np.ascontiguousarray(scalars, dtype=np.uint8)
    w = scalars.view("<u8")
    low = w.copy()
    low[:, 3] &= np.uint64(2**60 - 1)
    carry = _at_least(low, CARRY_EDGE)
    top = (w[:, 3] >> np.uint64(60)).astype(np.int64) + carry
    keep = top <= 8
    mag = _limbs(scalars)
    mag[15] = np.where(keep, mag[15], mag[15] & 0x0FFF)
    return mag, ~keep & carry


def effective_int(s: bytes) -> int:
    """The same rule for one scalar, on Python integers."""
    v = int.from_bytes(s, "little")
    low = v & (2**252 - 1)
    carry = int(low >= CARRY_EDGE)
    if (v >> 252) + carry <= 8:
        return v
    return low - 2**252 if carry else low


def expected(scalars, r, t):
    """Encoding of sum_i Point::mul(s_i, r_i*B + t_i*T8) for (n, 32) uint8 scalars and r, (n,) t."""
    n = scalars.shape[0]
    assert r.shape[0] == n and len(t) == n and n < (1 << 33)   # 2^33 blocks of < 2^50 stay below 2^63
    acc = np.zeros((16, 16), dtype=np.int64)                    # acc[j, k] = sum_i mag_i[j] * r_i[k]
    negr = np.zeros(16, dtype=np.int64)                         # limbs of the sum of r_i over negative eff
    for lo in range(0, n, _BLOCK):
        mag, neg = effective(scalars[lo:lo + _BLOCK])
        rl = _limbs(r[lo:lo + _BLOCK])
        acc += np.rint(mag.astype(np.float64) @ rl.T.astype(np.float64)).astype(np.int64)
        negr += rl[:, neg].sum(axis=1)
    k = sum(int(acc[j, i]) << (16 * (j + i)) for j in range(16) for i in range(16))
    k = (k - (sum(int(negr[i]) << (16 * i) for i in range(16)) << 252)) % L
    tors = int(((np.asarray(scalars[:, 0], dtype=np.int64) & 7) * np.asarray(t, dtype=np.int64)).sum()) % 8
    return O.point_encode(O.point_add(O._mul_int(k, O.BASE), O._mul_int(tors, _T8_PT)))


# ---- points with known discrete logs -------------------------------------------------------------------------------
def point_logs(n, seed):
    """(r, t): r pairwise distinct and below 2^252 (so below L; bytes 0..3 hold the index), t in 0..7."""
    rng = np.random.default_rng([seed, 0x5EED])
    r = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    r[:, 31] &= 0x0F
    r[:, :4] = np.arange(n, dtype="<u4").view(np.uint8).reshape(n, 4)
    t = rng.integers(0, 8, size=n, dtype=np.uint8)
    return r, t


def gpu_points(ctx, n, seed, coracle, sample=2048):
    """(encodings, r, t) with P_i = r_i*B + t_i*T8 computed by ctx (variable-time fixed-base multiplication, then
    point addition), and a random sample of them checked against the C oracle and the Python oracle."""
    from importlib import import_module

    kb = import_module("kyber-rs_b200")
    r, t = point_logs(n, seed)
    base = ctx.point_mul_base_batch(r, kb.binding.FLAG_VARTIME)
    pts, st = ctx.point_add_batch(base, TORSION[t])
    assert not st.any()
    idx = np.random.default_rng([seed, 1]).choice(n, size=min(n, sample), replace=False)
    want_b = coracle.mul_base_batch(r[idx], nthreads=8)
    assert (base[idx] == want_b).all()
    for i, b in zip(idx.tolist(), want_b):
        assert pts[i].tobytes() == O.point_encode(O.point_add(O.point_decode(b.tobytes()), O._mul_int(int(t[i]), _T8_PT)))
    return pts, r, t


def oracle_points(n, seed, coracle):
    """The same points built on the host with the C oracle."""
    r, t = point_logs(n, seed)
    base = coracle.mul_base_batch(r, nthreads=8)
    pts = np.frombuffer(b"".join(coracle.point_add(b.tobytes(), TORSION[k].tobytes()) for b, k in zip(base, t)), dtype=np.uint8).reshape(n, 32).copy()
    return pts, r, t


# ---- scalar families: each (n, seed[, c]) -> (n, 32) uint8 --------------------------------------------------------
def _rng(seed, tag):
    return np.random.default_rng([seed, tag])


def uniform(n, seed):
    """Raw 256-bit scalars: top nibbles 9..15 included, so about half have a negative or truncated effective scalar."""
    return _rng(seed, 1).integers(0, 256, size=(n, 32), dtype=np.uint8)


def reduced(n, seed):
    """Scalars below L: 252 random bits (what reduction mod L gives but for a 2^-125 fraction), plus L-1-k at a few
    positions.  The top windows hold one or two buckets, whose runs span many accumulation threads."""
    s = _rng(seed, 2).integers(0, 256, size=(n, 32), dtype=np.uint8)
    s[:, 31] &= 0x0F
    m = min(n, 7)
    s[np.linspace(0, n - 1, m).astype(np.int64)] = to_bytes([L - 1 - k for k in range(m)])
    return s


def equal(n, seed):
    return np.tile(_rng(seed, 3).integers(0, 256, size=(1, 32), dtype=np.uint8), (n, 1))


def sparse(n, seed):
    """Mostly zero: about one scalar in 1000 is a random raw scalar."""
    rng = _rng(seed, 4)
    s = np.zeros((n, 32), dtype=np.uint8)
    idx = rng.choice(n, size=max(1, n // 1000), replace=False)
    s[idx] = rng.integers(0, 256, size=(idx.shape[0], 32), dtype=np.uint8)
    return s


def small(n, seed, c):
    """1..2^c: only window 0 holds a digit (2^c itself carries into window 1)."""
    v = _rng(seed, 5).integers(1, (1 << c) + 1, size=n, dtype=np.int64)
    s = np.zeros((n, 32), dtype=np.uint8)
    s[:, :8] = v.astype("<u8").view(np.uint8).reshape(n, 8)
    return s


def carry_chain(n, seed, c):
    """Every c-bit digit below bit 252 is half or half + 1 (half = 2^(c-1)): each half + 1 becomes a negative digit
    and carries, so the signed-digit carry runs through all windows.  Below 2^252, so the magnitude is s itself."""
    bits = np.zeros((n, 256), dtype=np.uint8)
    for w in range(0, 252, c):
        if w + c - 1 < 252:
            bits[:, w + c - 1] = 1
        bits[:, w] |= _rng(seed, 6 + w).integers(0, 2, size=n, dtype=np.uint8)
    return np.packbits(bits, axis=1, bitorder="little")


def edge_values():
    vals = [0, 1, 8, L, L - 1, L + 1, 8 * L, 2**252, 2**252 - 1, 2**253 - 1, 2**255, 2**255 - 1, 2**256 - 1,
            int("88" * 32, 16), int("77" * 31 + "f7", 16), int("7" * 63 + "8", 16), int("8" * 63 + "7", 16)]
    for top in (0, 1, 8, 9, 15):          # the carry boundary of the effective scalar under each top-nibble class
        for d in (-1, 0, 1):
            vals.append((top << 252) + CARRY_EDGE + d)
    return vals


EDGES = to_bytes(edge_values())


def edges(n, seed):
    """Every edge scalar, cycled to n in a shuffled order."""
    s = np.tile(EDGES, ((n + EDGES.shape[0] - 1) // EDGES.shape[0], 1))[:n]
    return s[_rng(seed, 7).permutation(n)].copy() if n >= EDGES.shape[0] else s.copy()


FAMILIES = {
    "uniform": lambda n, seed, c: uniform(n, seed),
    "reduced": lambda n, seed, c: reduced(n, seed),
    "equal": lambda n, seed, c: equal(n, seed),
    "sparse": lambda n, seed, c: sparse(n, seed),
    "small": small,
    "carry": carry_chain,
    "edges": lambda n, seed, c: edges(n, seed),
}
