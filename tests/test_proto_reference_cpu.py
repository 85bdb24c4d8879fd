"""The exact protocol references of tests/proto_reference.py against the oracle's restatement of the reference
(oracle/ed25519_bigint.py, and the C oracle for the challenge hash) at small sizes, and the index sets they run at.
CPU only; the GPU counterpart is tests/test_gpu_proto_shapes.py."""
import numpy as np
import pytest

import proto_reference as P
from oracle import ed25519_bigint as O

L = O.L


def _pt(v):
    return O._mul_int(v, O.BASE)


def test_index_set():
    """Distinct, unsorted, deterministic; every special index once k reaches them; the NAFs and node spacings they
    stand for: 33-digit NAFs (x = 2^32, 2^32 - 1), the densest 33-digit NAF, adjacent nodes and nodes 2^31 apart."""
    for k in (1, 2, 5, len(P.SPECIAL), 683, 2048):
        s = P.index_set(k, seed=k)
        assert s.dtype == np.uint32 and len(s) == k == len(set(s.tolist()))
        assert (s == P.index_set(k, seed=k)).all()
        assert set(s.tolist()) >= set(P.SPECIAL[:k])
        if k >= 5:
            assert (np.diff(s.astype(np.int64)) < 0).any() and (np.diff(s.astype(np.int64)) > 0).any()
    assert set(P.index_set(2, seed=0).tolist()) == {2**32 - 1, 2**31 - 1}
    sp = set(P.SPECIAL)
    assert {a for a in sp if a + 1 in sp} >= {0, 1, 2**31 - 1, 2**32 - 2, 0x55555554, 0xAAAAAAA9}
    assert {a for a in sp if a + 2**31 in sp} >= {0, 2**31 - 1, 0x2AAAAAAA, 0x55555555}
    nafs = {i: P.naf(i + 1) for i in P.SPECIAL}
    assert len(nafs[2**32 - 1]) == len(nafs[2**32 - 2]) == len(nafs[0xAAAAAAAA]) == 33
    assert sum(d != 0 for d in nafs[0xAAAAAAAA]) == 17
    rng = np.random.default_rng(1)
    for x in [i + 1 for i in P.SPECIAL] + rng.integers(1, 2**32 + 1, size=2000).tolist():
        d = P.naf(x)
        assert sum(v << j for j, v in enumerate(d)) == x and d[-1] == 1 and len(d) <= 33
        assert all(d[j] == 0 or d[j + 1] == 0 for j in range(len(d) - 1))


def test_to_ints_roundtrip():
    v = [0, 1, L - 1, L, 2**256 - 1, 2**255 + 19, 2**64, 2**64 - 1] + P.scalars(50, 1)
    assert P.to_ints(P.to_bytes(v)) == v
    assert all(0 <= s < L for s in P.scalars(1000, 2))


@pytest.mark.parametrize("t", [1, 2, 5, 9])
def test_poly_eval_matches_pripoly_eval(t):
    """poly_eval(coeffs, i + 1) is PriPoly::eval at index i, for 32-bit indices and unreduced coefficients."""
    coeffs = P.scalars(t, 10 + t)
    if t > 1:
        coeffs[-1] = 2**256 - 1
    idx = P.index_set(24, seed=t).tolist()
    cb = [c.to_bytes(32, "little") for c in coeffs]
    many = P.poly_eval_many(coeffs, [i + 1 for i in idx])
    for i, v in zip(idx, many):
        assert P.poly_eval(coeffs, i + 1) == v == int.from_bytes(O.pripoly_eval(cb, i), "little")


def test_pubpoly_eval_is_poly_eval_times_base():
    """PubPoly::eval of the commitments c_j * B at index i is poly_eval(c, i + 1) * B (the oracle's full scalar mults)."""
    coeffs = P.scalars(3, 20)
    commits = [_pt(c) for c in coeffs]
    for i in (0, 2**31 - 1, 2**32 - 1):
        assert O.point_eq(O.pubpoly_eval(commits, i), _pt(P.poly_eval(coeffs, i + 1)))


@pytest.mark.parametrize("k", [1, 2, 3, 5])
def test_lagrange_at_zero_matches_recover_commit(k):
    """sum_i lam_i y_i is the discrete log of recover_commit's interpolation of the points y_i * B, over 32-bit nodes."""
    idx = P.index_set(k, seed=30 + k).tolist()
    lam = P.lagrange_at_zero([i + 1 for i in idx])
    ys = P.scalars(k, 31 + k)
    want = O.recover_commit([(i, _pt(y)) for i, y in zip(idx, ys)])
    assert O.point_eq(want, _pt(P.weighted_sum(lam, ys)))


@pytest.mark.parametrize("k", [1, 7, 64])
def test_lagrange_at_zero_recovers_the_secret(k):
    """On every node set, the weights give p(0) for polynomials of degree below k, and not for degree k."""
    for seed, idx in enumerate((P.index_set(k, seed=k), P.small_index_set(k, 1024, seed=k))):
        xs = [int(i) + 1 for i in idx]
        lam = P.lagrange_at_zero(xs)
        coeffs = P.scalars(k, 40 + seed)
        assert P.weighted_sum(lam, P.poly_eval_many(coeffs, xs)) == coeffs[0]
        over = coeffs + [1]
        assert P.weighted_sum(lam, P.poly_eval_many(over, xs)) != over[0]


def test_lagrange_basis_and_recover_pub_poly():
    """The constant term of the oracle's lagrange_basis_j is lam_j, and recover_pub_poly over points poly_eval(c, x) * B
    gives back the commitments c_j * B."""
    for k in (1, 2, 3):
        idx = P.index_set(k, seed=50 + k).tolist()
        xs = {i: O.scalar_set_int64(i + 1) for i in idx}
        lam = P.lagrange_at_zero([i + 1 for i in idx])
        for j, i in enumerate(idx):
            assert int.from_bytes(O.lagrange_basis(i, xs)[0], "little") == lam[j]
        coeffs = P.scalars(k, 51 + k)
        got = O.recover_pub_poly([(i, _pt(P.poly_eval(coeffs, i + 1))) for i in idx])
        assert [O.point_encode(p) for p in got] == [O.point_encode(_pt(c)) for c in coeffs]


@pytest.mark.parametrize("msg_len", [0, 1, 47, 48, 111, 112, 175, 176, 1023])
def test_challenge_matches_dss_hash_sig(coracle, msg_len):
    """SHA-512(R || A || msg) mod L is hash_sig at the padding edges of a 64-byte prefix (64 + len = 111 / 112 mod 128),
    against the Python oracle and the C oracle's own SHA-512."""
    rng = np.random.default_rng(msg_len)
    r, a = _pt(P.scalars(1, 60 + msg_len)[0] + 5), _pt(P.scalars(1, 61 + msg_len)[0] + 7)
    msg = rng.integers(0, 256, size=msg_len, dtype=np.uint8).tobytes()
    h = P.challenge(O.point_encode(r), O.point_encode(a), msg)
    assert h.to_bytes(32, "little") == O.dss_hash_sig(r, a, msg)
    rb = np.frombuffer(O.point_encode(r), dtype=np.uint8).reshape(1, 32)
    ab = np.frombuffer(O.point_encode(a), dtype=np.uint8).reshape(1, 32)
    assert coracle.dss_hash_sig(rb, ab, msg) == h.to_bytes(32, "little")


def test_session_id_matches_oracle():
    for nd, n, t in ((1, 1, 1), (2, 5, 3)):
        pts = [_pt(s + 1) for s in P.scalars(nd + n + nd * t, 70 + n)]
        enc = np.frombuffer(b"".join(O.point_encode(p) for p in pts), dtype=np.uint8).reshape(-1, 32)
        for d in range(nd):
            com = nd + n + d * t
            want = O.session_id(pts[d], pts[nd:nd + n], pts[com:com + t], t)
            assert P.session_id(enc[d], enc[nd:nd + n], enc[com:com + t], t) == want
