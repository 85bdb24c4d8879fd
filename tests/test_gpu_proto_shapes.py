"""The protocol entry points (csrc/capi_proto.cu, proto.cuh, poly.cuh, the PubPoly / PriPoly paths of capi_poly.cu)
at the full DKG shape (n = 1024, t = 683) and at 32-bit share indices, against the exact integers of
tests/proto_reference.py.  Every expected point is (exact scalar) * B from the C oracle; inputs the device reads
(commitments, public shares) come from the context's fixed-base multiplication, which test_gpu_parity.py holds
bit-exact.  Needs a B200."""
import importlib
import os

import numpy as np
import pytest

import proto_reference as P
from helpers import _off_curve
from oracle import ed25519_bigint as O

pytestmark = pytest.mark.gpu

L = P.L
NTHREADS = os.cpu_count() or 8
T8 = O.WEAK_KEYS[2]                       # encoding of a point of order 8
TOP = 2**32 - 1                           # the largest index: x = 2^32


@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


@pytest.fixture(scope="module")
def ctx(kb):
    c = kb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def lagrange():
    """Lagrange weights at zero per node set, computed once."""
    cache = {}

    def get(idx):
        key = np.asarray(idx, dtype=np.uint32).tobytes()
        if key not in cache:
            cache[key] = P.lagrange_at_zero([int(i) + 1 for i in idx])
        return cache[key]

    return get


def _xs(idx):
    return [int(i) + 1 for i in idx]


def _times_base(coracle, vals):
    """(exact scalar) * B for each value, from the C oracle."""
    return coracle.mul_base_batch(P.to_bytes(vals), nthreads=NTHREADS)


def _points(ctx, vals):
    return ctx.point_mul_base_batch(P.to_bytes(vals))


def _with_torsion(p32, x):
    """p + x * T8 for an encoding p, exactly (x only matters mod 8)."""
    return O.point_encode(O.point_add(O.point_decode(bytes(p32)), O._mul_int(x % 8, O.point_decode(T8))))


# ---- 1. recover_commit ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ncols", [1, 8])
@pytest.mark.parametrize("k", [1, 2, 683, 1023, 2048])
def test_recover_commit_batch(ctx, coracle, lagrange, k, ncols):
    """ncols columns of k public shares at the extreme indices interpolate to p_c(0) * B; the same under a
    permutation of the rows; an undecodable share flags its column and no other.  Column 0 holds shares of a
    polynomial of degree min(k, 4) - 1, so its answer is that polynomial's secret; the other columns hold random
    shares, whose interpolant at zero is sum_i lam_i y_i."""
    idx = P.index_set(k, seed=k)
    xs = _xs(idx)
    lam = lagrange(idx)
    poly0 = P.scalars(min(k, 4), 10000 + k)
    ys = [P.poly_eval_many(poly0, xs)] + [P.scalars(k, 100 * c + k) for c in range(1, ncols)]
    secrets = [P.weighted_sum(lam, y) for y in ys]
    assert secrets[0] == poly0[0]
    want = _times_base(coracle, secrets)
    pts = _points(ctx, [v for y in ys for v in y])              # [column][share]
    got, st = ctx.recover_commit_batch(idx, pts, ncols=ncols)
    assert not st.any() and (got == want).all(), np.nonzero((got != want).any(axis=1))[0]
    perm = np.random.default_rng(k).permutation(k)
    got, st = ctx.recover_commit_batch(idx[perm], pts.reshape(ncols, k, 32)[:, perm].reshape(-1, 32), ncols=ncols)
    assert not st.any() and (got == want).all(), "permuted rows"
    col = ncols - 1
    bad = pts.copy()
    bad[col * k + k // 2] = np.frombuffer(_off_curve(k), dtype=np.uint8)
    got, st = ctx.recover_commit_batch(idx, bad, ncols=ncols)
    assert st.tolist() == [int(c == col) for c in range(ncols)]
    assert (got[:col] == want[:col]).all()


# ---- 2. recover_pub_poly -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [172, 256, 683, 1022, 1023])
def test_recover_pub_poly(ctx, coracle, k):
    """k public shares p(x_j) * B at the extreme indices give back every commitment coeff_c * B: k_lagrange_basis
    runs as one block of k + 1 threads, up to the 1024 of its launch bounds."""
    idx = P.index_set(k, seed=k)
    coeffs = P.scalars(k, 200 + k)
    pub = _points(ctx, P.poly_eval_many(coeffs, _xs(idx)))
    got, st = ctx.recover_pub_poly(idx, pub)
    want = _times_base(coracle, coeffs)
    assert not st.any() and (got == want).all(), np.nonzero((got != want).any(axis=1))[0][:16]


def test_interpolation_rejects_what_it_cannot_interpolate(kb, ctx):
    """recover_pub_poly at k = 1024 (more threads than one block holds) and every interpolation entry with a repeated
    index (a zero denominator) raise instead of computing."""
    idx = P.index_set(1024, seed=1024)
    pts = _points(ctx, P.scalars(1024, 7))
    with pytest.raises(kb.KBError):
        ctx.recover_pub_poly(idx, pts)
    dup = idx[:683].copy()
    dup[600] = dup[5]
    with pytest.raises(kb.KBError):
        ctx.recover_pub_poly(dup, pts[:683])
    with pytest.raises(kb.KBError):
        ctx.recover_commit_batch(dup, pts[:683])
    with pytest.raises(kb.KBError):
        ctx.dkg_resharing_key(1, dup, pts[:683])


# ---- 3. resharing_key ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def reshare(ctx):
    """683 qualified nodes' deals of 683 commitments each, f[i][c] * B (node-major, as dkg_resharing_key takes them)."""
    k = new_t = 683
    f = np.array(P.scalars(k * new_t, 300), dtype=object).reshape(k, new_t)
    return f, _points(ctx, f.reshape(-1).tolist())


@pytest.mark.parametrize("nodes", ["below-1024", "extreme"])
def test_dkg_resharing_key(ctx, coracle, lagrange, reshare, nodes):
    """resharing_key at the DKG shape (new_t = 683 columns over k = 683 qualified nodes): commitment c is
    (sum_i lam_i f[i][c]) * B exactly, and the check of the new share at share_idx = 0, 1023, 2^32 - 1 accepts the
    honest share and rejects it plus one."""
    k = new_t = 683
    f, coeffs = reshare
    idx = P.small_index_set(k, 1024, seed=3) if nodes == "below-1024" else P.index_set(k, seed=3)
    lam = np.array(lagrange(idx), dtype=object)
    F = [int(v) % L for v in lam.dot(f)]
    want = _times_base(coracle, F)
    out, st, chk = ctx.dkg_resharing_key(new_t, idx, coeffs)
    assert not st.any() and chk is None and (out == want).all(), np.nonzero((out != want).any(axis=1))[0][:16]
    for share_idx in (0, 1023, TOP):
        s = P.poly_eval(F, share_idx + 1)
        for share, ok in ((s, True), ((s + 1) % L, False)):
            out2, _, chk = ctx.dkg_resharing_key(new_t, idx, coeffs, share_idx=share_idx, share=P.to_bytes([share])[0])
            assert chk is ok, (share_idx, ok)
            assert (out2 == want).all()


# ---- 4. PubPoly::eval and the VSS share check ----------------------------------------------------------------------
@pytest.mark.parametrize("t", [1, 2, 683, 1024])
def test_pubpoly_eval_and_verify_deals(ctx, coracle, t):
    """Two polynomials evaluated at 64 extreme indices each (every special index among them): p(x) * B exactly;
    the share check accepts p(x) and rejects p(x) + 1.  With a point of order 8 added to coefficient 1, the
    evaluation is p(x) * B + x * T8, and the check of the honest share passes iff 8 | x: at x = 2^32 it passes,
    at x = 2^32 - 1 it fails."""
    npoly, nidx = 2, 64
    idx1 = P.index_set(nidx, seed=400 + t)
    coeffs = [P.scalars(t, 400 + 2 * t + d) for d in range(npoly)]
    commits = _points(ctx, coeffs[0] + coeffs[1])
    poly_id = np.repeat(np.arange(npoly, dtype=np.uint32), nidx)
    idx = np.tile(idx1, npoly)
    vals = [v for d in range(npoly) for v in P.poly_eval_many(coeffs[d], _xs(idx1))]
    want = _times_base(coracle, vals)
    got, st = ctx.pubpoly_eval_batch(commits, t, poly_id, idx)
    assert not st.any() and (got == want).all(), idx[(got != want).any(axis=1)]
    shares = P.to_bytes(vals)
    verdict_want = np.ones(npoly * nidx, dtype=np.uint8)
    for k in [int(np.nonzero(idx1 == TOP)[0][0]), nidx + int(np.nonzero(idx1 == 0)[0][0]), nidx + 7]:
        shares[k] = P.to_bytes([(vals[k] + 1) % L])[0]
        verdict_want[k] = 0
    verdict = ctx.vss_verify_deals_batch(commits, t, poly_id, idx, shares)
    assert (verdict == verdict_want).all(), idx[verdict != verdict_want]
    if t < 2:
        return
    tc = commits.copy()
    tc[t + 1] = np.frombuffer(_with_torsion(commits[t + 1], 1), dtype=np.uint8)
    sel = np.array([TOP, 2**32 - 2, 7, 0x55555555, 2**31 - 1], dtype=np.uint32)   # x = 2^32, 2^32 - 1, 8, 0x55555556, 2^31
    x = _xs(sel)
    v1 = P.poly_eval_many(coeffs[1], x)
    pid = np.ones(len(sel), dtype=np.uint32)
    got, st = ctx.pubpoly_eval_batch(tc, t, pid, sel)
    assert not st.any()
    assert [g.tobytes() for g in got] == [_with_torsion(p, xx) for p, xx in zip(_times_base(coracle, v1), x)]
    verdict = ctx.vss_verify_deals_batch(tc, t, pid, sel, P.to_bytes(v1))
    assert verdict.tolist() == [1, 0, 1, 0, 1]


# ---- 5. PriPoly::eval at the cfg4 shape ----------------------------------------------------------------------------
def test_pripoly_eval_cfg4_shape(ctx):
    """1024 polynomials of 683 raw 256-bit coefficients (most of them not reduced) at indices 0..1023: the full rows
    of dealers 0, 1, 511, 1023 and index 1023 of every dealer, exactly mod L."""
    npoly, t, n = 1024, 683, 1024
    raw = np.random.default_rng(5).integers(0, 256, size=(npoly * t, 32), dtype=np.uint8)
    raw[0] = 0xFF
    raw[t - 1] = np.frombuffer(L.to_bytes(32, "little"), dtype=np.uint8)
    got = ctx.pripoly_eval_batch(raw, t, n)
    assert got.shape == (npoly * n, 32)
    c = np.array(P.to_ints(raw), dtype=object).reshape(npoly, t)
    xs = list(range(1, n + 1))
    for d in (0, 1, 511, 1023):
        want = P.to_bytes(P.poly_eval_many(c[d].tolist(), xs))
        assert (got[d * n:(d + 1) * n] == want).all(), (d, np.nonzero((got[d * n:(d + 1) * n] != want).any(axis=1))[0][:8])
    v = np.zeros(npoly, dtype=object)
    for j in range(t - 1, -1, -1):
        v = (v * n + c[:, j]) % L
    col = got[np.arange(npoly) * n + (n - 1)]
    want = P.to_bytes(v.tolist())
    assert (col == want).all(), np.nonzero((col != want).any(axis=1))[0][:8]


# ---- 6. DSS partial signatures -------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dss(ctx):
    """t = 683, m = 1024 partials: 1000 distinct extreme indices, 24 of them repeated (x = 2^32 among them), all in
    a random order; the two polynomials evaluated at every item."""
    t, m = 683, 1024
    rng = np.random.default_rng(6)
    base = P.index_set(1000, seed=6)
    rep = np.concatenate([[TOP, 0], rng.choice(base[~np.isin(base, [TOP, 0])], size=22, replace=False)]).astype(np.uint32)
    idx = np.concatenate([base, rep])[rng.permutation(m)]
    rc, lc = P.scalars(t, 61), P.scalars(t, 62)
    rcom, lcom = _points(ctx, rc), _points(ctx, lc)
    xs = _xs(idx)
    return rcom, lcom, idx, P.poly_eval_many(rc, xs), P.poly_eval_many(lc, xs)


@pytest.mark.parametrize("msg_len", [0, 1, 47, 48, 111, 112, 175, 176, 1023, 1 << 20])
def test_dss_verify_partials(ctx, coracle, dss, msg_len):
    """The challenge SHA-512(R || A || msg) mod L at the padding edges of its 64-byte prefix and for a 1 MiB message,
    and the verdicts of 1024 partials (honest 1, corrupted 0, one of two copies of x = 2^32 corrupted); at 1023 bytes
    a 256-item selection is also held to the C oracle's full scalar multiplications."""
    rcom, lcom, idx, rv, lv = dss
    msg = np.random.default_rng(msg_len).integers(0, 256, size=msg_len, dtype=np.uint8).tobytes()
    h = P.challenge(rcom[0], lcom[0], msg)
    vals = [(r + h * l) % L for r, l in zip(rv, lv)]
    want = np.ones(len(idx), dtype=np.uint8)
    top = np.nonzero(idx == TOP)[0]
    assert len(top) == 2
    for k in (int(top[0]), 0, len(idx) - 1, 500 + msg_len % 17):
        vals[k] = (vals[k] + 1 + msg_len) % L
        want[k] = 0
    partials = P.to_bytes(vals)
    got, hs = ctx.dss_verify_partials(rcom, lcom, msg, idx, partials)
    assert hs == h.to_bytes(32, "little")
    assert (got == want).all(), idx[got != want]
    if msg_len == 1023:
        must = np.unique(np.concatenate([np.nonzero(np.isin(idx, P.SPECIAL))[0], np.nonzero(want == 0)[0]]))
        sel = np.concatenate([must, np.setdiff1d(np.arange(len(idx)), must)[:256 - len(must)]])
        assert (coracle.dss_partial_batch(rcom, lcom, msg, idx[sel], partials[sel], nthreads=NTHREADS) == got[sel]).all()


# ---- 7. session ids ------------------------------------------------------------------------------------------------
def test_vss_session_ids_dkg_shape(ctx, coracle):
    """4 dealers, 1024 verifiers, 683 commitments each: SHA-256 over the encodings, from 32-byte and raw-limb inputs."""
    nd, n, t = 4, 1024, 683
    pts = _points(ctx, P.scalars(nd + n + nd * t, 700))
    dealers, verifiers, commits = pts[:nd], pts[nd:nd + n], pts[nd + n:]
    want = [P.session_id(dealers[d], verifiers, commits[d * t:(d + 1) * t], t) for d in range(nd)]
    got, st = ctx.vss_session_ids(dealers, verifiers, commits, t)
    assert not st.any() and [g.tobytes() for g in got] == want
    limbs = [np.stack([coracle.point_limbs(p.tobytes()) for p in a]) for a in (dealers, verifiers, commits)]
    got, st = ctx.vss_session_ids(*limbs, t, limbs=True)
    assert not st.any() and [g.tobytes() for g in got] == want
