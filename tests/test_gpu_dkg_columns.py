"""kb_dkg_verify_columns: the share checks of a DKG round for a range of verifiers (dkgcol.cuh).  Every case compares the
verdicts item by item with kb_vss_verify_deals_batch on the same items (poly_id = d, idx = i), samples them against the
oracle, and checks both round-check modes (a partial range reports no fallback) and both planner routes."""
import contextlib
import importlib
import os
import subprocess

import numpy as np
import pytest

from helpers import ROOT, xof_bytes
from oracle import ed25519_bigint as O

pytestmark = pytest.mark.gpu

L = O.L


@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


@contextlib.contextmanager
def _context(kb, mode="exact", columns=None):
    """A context in the given round-check mode; columns = "0" / "1" forces the per-share / column route (KB_DKG_COLUMNS)."""
    old = os.environ.get("KB_DKG_COLUMNS")
    if columns is not None:
        os.environ["KB_DKG_COLUMNS"] = columns
    try:
        c = kb.Context(0)
    finally:
        if old is None:
            os.environ.pop("KB_DKG_COLUMNS", None)
        else:
            os.environ["KB_DKG_COLUMNS"] = old
    c.set_round_check(mode)
    try:
        yield c
    finally:
        c.close()


@pytest.fixture(scope="module")
def ctxs(kb):
    """(exact, batched, column route forced, per-share route forced)"""
    with _context(kb) as e, _context(kb, "batched") as b, _context(kb, "exact", "1") as col, _context(kb, "batched", "0") as per:
        yield e, b, col, per


def _coeffs(tag, nd, t):
    c = np.frombuffer(xof_bytes(f"cols/{tag}", 32 * nd * t), dtype=np.uint8).reshape(nd * t, 32).copy()
    c[:, 31] &= 0x0F
    return c


def _round(ctx, n, t, nd, tag):
    """Commitments and the honest shares of nd dealers for every verifier 0..n-1 ([d * n + i])."""
    coeffs = _coeffs(tag, nd, t)
    return ctx.point_mul_base_batch(coeffs, 1).copy(), ctx.pripoly_eval_batch(coeffs, t, n).copy()


def _shares_at(coeffs, t, nd, xs):
    """Honest shares f_d(x) mod L for the given x (Python integers), [d * len(xs) + c]."""
    out = np.zeros((nd * len(xs), 32), dtype=np.uint8)
    for d in range(nd):
        a = [int.from_bytes(coeffs[d * t + j].tobytes(), "little") for j in range(t)]
        for c, x in enumerate(xs):
            v = 0
            for cj in reversed(a):
                v = (v * x + cj) % L
            out[d * len(xs) + c] = np.frombuffer(v.to_bytes(32, "little"), dtype=np.uint8)
    return out


def _cols(shares, n, dlo, dhi, lo, hi):
    return shares.reshape(-1, n, 32)[dlo:dhi, lo:hi].reshape(-1, 32).copy()


def _reference(ctx, commits, t, dlo, dhi, lo, hi, sh):
    k = hi - lo
    pid = np.repeat(np.arange(dlo, dhi, dtype=np.uint32), k)
    idx = np.tile(np.arange(lo, hi, dtype=np.uint64), dhi - dlo).astype(np.uint32)
    return ctx.vss_verify_deals_batch(commits, t, pid, idx, sh)


def _check(ctxs, n, t, commits, sh, dlo, dhi, lo, hi, fmt=0, want=None):
    """Every context gives the reference verdicts (or want); a partial range reports 0 fallbacks.  Returns the verdicts."""
    if want is None:
        want = _reference(ctxs[0], commits, t, dlo, dhi, lo, hi, sh)
    for c in ctxs:
        got = c.dkg_verify_columns(n, t, commits, sh, lo, hi, dealer_lo=dlo, dealer_hi=dhi, fmt=fmt)
        assert (got == want).all(), (lo, hi, dlo, dhi, np.argwhere(got != want)[:8])
        if not (lo == 0 and hi == n):
            assert c.round_fallbacks() == 0
    return want


def _oracle_sample(commits, t, d, i, share):
    pts = [O.point_decode(commits[d * t + j].tobytes()) for j in range(t)]
    if any(p is None for p in pts):
        return 0
    return int(O.pubpoly_check(pts, i, share.tobytes()))


def _add_point(ctx, enc, p):
    return ctx.point_add_batch(enc.reshape(1, 32), np.frombuffer(p, dtype=np.uint8).reshape(1, 32))[0][0]


def _torsion(order):
    t8 = O.point_decode(O.WEAK_KEYS[2])
    return O.point_encode(O._mul_int(8 // order, t8))


@pytest.mark.parametrize("k", [1, 2, 7, 64])
def test_ranges_small_round(ctxs, k):
    """n = 64, t = 43, 16 dealers with wrong shares and a torsion dealer: k columns at ver_lo = 0, 1, n - k, and dealer
    sub-ranges; the full range equals kb_dkg_verify_round in both modes."""
    e = ctxs[0]
    n, t, nd = 64, 43, 16
    commits, shares = _round(e, n, t, nd, "small")
    commits[5 * t + 1] = _add_point(e, commits[5 * t + 1], _torsion(8))
    for d, i in ((0, 0), (3, 1), (3, 62), (9, 63), (15, 30)):
        shares[d * n + i, 4] ^= 0x10
    for lo in sorted({0, min(1, n - k), n - k}):
        for dlo, dhi in ((0, nd), (3, 9)):
            _check(ctxs, n, t, commits, _cols(shares, n, dlo, dhi, lo, lo + k), dlo, dhi, lo, lo + k)
    if k == 64:
        for c in ctxs[:2]:
            assert (c.dkg_verify_columns(n, t, commits, shares, 0, n) == c.dkg_verify_round(n, t, commits, shares)).all()
    d, i = 5, 7   # x = 8: the order-8 point vanishes
    sh = _cols(shares, n, d, d + 1, i, i + 1)
    assert e.dkg_verify_columns(n, t, commits, sh, i, i + 1, dealer_lo=d, dealer_hi=d + 1)[0] == _oracle_sample(commits, t, d, i, sh[0]) == 1


def test_full_range_reports_the_round(ctxs, kb):
    """ver_lo = 0, ver_hi = n is kb_dkg_verify_round itself: the same verdicts and, in BATCHED mode, its fallback count."""
    e, b = ctxs[0], ctxs[1]
    n, t, nd = 48, 5, 6
    commits, shares = _round(e, n, t, nd, "full")
    shares[2 * n + 9, 0] ^= 1
    want = e.dkg_verify_round(n, t, commits, shares)
    assert (b.dkg_verify_columns(n, t, commits, shares, 0, n) == want).all()
    assert b.round_fallbacks() == 1
    assert (b.dkg_verify_columns(n, t, commits, _cols(shares, n, 0, nd, 0, n - 1), 0, n - 1) == want.reshape(nd, n)[:, :n - 1].ravel()).all()
    assert b.round_fallbacks() == 0


def test_cfg4_shape(ctxs):
    """n = 1 024, t = 683, 1 024 dealers: k = 1, 7 and 64 columns at several offsets, with wrong shares and a torsion dealer."""
    e = ctxs[0]
    n, t, nd = 1024, 683, 1024
    commits, shares = _round(e, n, t, nd, "cfg4")
    commits[700 * t + 2] = _add_point(e, commits[700 * t + 2], _torsion(4))
    rng = np.random.default_rng(4)
    for _ in range(40):
        d, i = rng.integers(0, nd), rng.integers(0, n)
        shares[d * n + i, 17] ^= 0x40
    for k, lo in ((1, 0), (1, 511), (1, n - 1), (7, 1), (7, 1000), (64, 0), (64, 333), (64, n - 64)):
        _check(ctxs, n, t, commits, _cols(shares, n, 0, nd, lo, lo + k), 0, nd, lo, lo + k)


@pytest.mark.parametrize("k", [1, 2, 7])
def test_32bit_indices(ctxs, k):
    """n = 2^32: the last k verifiers (x up to 2^32) and a range across 2^31, against the reference and the oracle."""
    e = ctxs[0]
    n, t, nd = 1 << 32, 43, 8
    coeffs = _coeffs("u32", nd, t)
    commits = e.point_mul_base_batch(coeffs, 1).copy()
    commits[3 * t] = _add_point(e, commits[3 * t], _torsion(2))
    for lo in (n - k, (1 << 31) - 1):
        xs = [lo + c + 1 for c in range(k)]
        sh = _shares_at(coeffs, t, nd, xs)
        sh[nd * k // 2, 3] ^= 2
        v = _check(ctxs, n, t, commits, sh, 0, nd, lo, lo + k)
        for d, c in ((0, k - 1), (3, 0), (nd // 2, 0)):
            assert v[d * k + c] == _oracle_sample(commits, t, d, lo + c, sh[d * k + c]), (lo, d, c)


@pytest.mark.parametrize("t", [1, 2, 3, 43, 683])
def test_thresholds(ctxs, t):
    e = ctxs[0]
    n, nd = 40, 6
    commits, shares = _round(e, n, t, nd, f"t{t}")
    shares[nd * n // 2 + 4, 8] ^= 1
    for lo, k in ((0, 1), (3, 5), (n - 7, 7)):
        _check(ctxs, n, t, commits, _cols(shares, n, 0, nd, lo, lo + k), 0, nd, lo, lo + k)


@pytest.mark.parametrize("t", [3, 5])
def test_torsion_every_residue(ctxs, t):
    """Points of order 2, 4 and 8 on coefficients 0, 1, 2 and t - 1 (one dealer each), x = 1 .. 8 and 14 .. 21."""
    e = ctxs[0]
    n = 24
    cases = [(o, j) for o in (2, 4, 8) for j in sorted({0, 1, 2, t - 1})]
    nd = len(cases)
    commits, shares = _round(e, n, t, nd, f"tor{t}")
    for d, (o, j) in enumerate(cases):
        commits[d * t + j] = _add_point(e, commits[d * t + j], _torsion(o))
    for lo in (0, 13):
        sh = _cols(shares, n, 0, nd, lo, lo + 8)
        v = _check(ctxs, n, t, commits, sh, 0, nd, lo, lo + 8)
        assert v.any() and not v.all()
        for d in range(0, nd, 3):
            for c in (0, 3, 7):
                assert v[d * 8 + c] == _oracle_sample(commits, t, d, lo + c, sh[d * 8 + c]), (cases[d], lo + c)


def test_bad_commitments_both_formats(ctxs, coracle):
    """An undecodable encoding and inconsistent limbs give 0 in every column of their dealer."""
    e = ctxs[0]
    n, t, nd = 32, 7, 6
    commits, shares = _round(e, n, t, nd, "bad")
    commits[2 * t + 3] = np.frombuffer(b"\x02" + b"\x00" * 30 + b"\x80", dtype=np.uint8)
    assert O.point_decode(commits[2 * t + 3].tobytes()) is None
    sh = _cols(shares, n, 0, nd, 5, 12)
    v = _check(ctxs, n, t, commits, sh, 0, nd, 5, 12).reshape(nd, 7)
    assert not v[2].any() and v[[0, 1, 3, 4, 5]].all()
    good, _ = _round(e, n, t, nd, "bad")
    limbs = np.stack([coracle.point_limbs(c.tobytes()) for c in good])
    limbs[4 * t + 1, 7] += 1   # T Z != X Y
    want = _reference(e, good, t, 0, nd, 5, 12, sh).reshape(nd, 7)
    assert want.all()
    want[4] = 0
    _check(ctxs, n, t, limbs, sh, 0, nd, 5, 12, fmt=1, want=want.ravel())


def test_share_forms(ctxs):
    """s + L, byte 31 > 127 and one wrong share per column, against the reference and the oracle."""
    e = ctxs[0]
    n, t, nd, lo, k = 64, 4, 8, 20, 8
    commits, shares = _round(e, n, t, nd, "forms")
    sh = _cols(shares, n, 0, nd, lo, lo + k)
    forms = {}
    for c in range(k):
        d = c % nd
        s = int.from_bytes(sh[d * k + c].tobytes(), "little")
        new = (s + L, s + (1 << 255), s + L + (1 << 255), (s + 1) % L)[c % 4]
        sh[d * k + c] = np.frombuffer(new.to_bytes(32, "little"), dtype=np.uint8)
        forms[(d, c)] = new
    v = _check(ctxs, n, t, commits, sh, 0, nd, lo, lo + k)
    for (d, c), _ in forms.items():
        assert v[d * k + c] == _oracle_sample(commits, t, d, lo + c, sh[d * k + c]), (d, c)
    assert v[0 * k + 0] == 1   # s + L


def test_device_form_on_a_stream(ctxs, kb):
    """kb_dev_dkg_verify_columns on torch tensors and a non-default stream, for a dealer sub-range (pointers at its first
    dealer), both routes, equal to the host form."""
    import torch

    e, _, col, per = ctxs
    n, t, nd, dlo, dhi, lo, k = 96, 9, 12, 4, 11, 40, 16
    commits, shares = _round(e, n, t, nd, "dev")
    shares[5 * n + 41, 2] ^= 8
    sh = _cols(shares, n, dlo, dhi, lo, lo + k)
    want = e.dkg_verify_columns(n, t, commits, sh, lo, lo + k, dealer_lo=dlo, dealer_hi=dhi)
    s = torch.cuda.Stream()
    for c in (e, col, per):
        dc = torch.from_numpy(commits[dlo * t:dhi * t].copy()).cuda()
        ds = torch.from_numpy(sh).cuda()
        dv = torch.full((sh.shape[0],), 7, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            c.dev_dkg_verify_columns(n, t, dhi - dlo, dc, ds, dv, lo, lo + k)
            got = dv.cpu().numpy()
        s.synchronize()
        assert (got == want).all()
        assert c.round_fallbacks() == 0


def test_argument_errors(ctxs):
    e = ctxs[0]
    Lb = e.L
    n, t, nd = 16, 3, 2
    commits, shares = _round(e, n, t, nd, "args")
    sh = _cols(shares, n, 0, nd, 2, 6)
    v = np.zeros(sh.shape[0], dtype=np.uint8)
    cp, sp, vp = commits.ctypes.data, sh.ctypes.data, v.ctypes.data

    def call(n_=n, t_=t, dlo=0, dhi=nd, lo=2, hi=6, fmt=0, ctx=e.h):
        return Lb.kb_dkg_verify_columns(ctx, n_, t_, dlo, dhi, lo, hi, fmt, cp, sp, vp)

    assert call() == 0
    for bad in (dict(lo=6, hi=6), dict(lo=7, hi=6), dict(hi=n + 1, lo=n - 3), dict(dlo=2, dhi=1), dict(n_=(1 << 32) + 1, lo=0, hi=4), dict(fmt=2), dict(t_=0), dict(ctx=None)):
        assert call(**bad) == -1, bad
    assert call(dlo=1, dhi=1) == 0   # empty dealer range
    assert Lb.kb_dkg_verify_columns(e.h, n, t, 0, nd, 2, 6, 0, None, sp, vp) == -1
    assert Lb.kb_dev_dkg_verify_columns(e.h, n, t, 0, 2, 6, 0, None, None, None, None) == 0
    assert Lb.kb_dev_dkg_verify_columns(e.h, n, t, nd, 6, 2, 0, None, None, None, None) == -1
    assert Lb.kb_dev_dkg_verify_columns(e.h, n, t, nd, 2, 6, 0, None, None, None, None) == -1
    assert call(n_=1 << 32, lo=(1 << 32) - 4, hi=1 << 32) == 0


def test_columns_from_plain_c(kb, ctxs, tmp_path):
    """tests/c/dkg_columns_check.c: verdicts in both modes, fallback count 0 and argument errors from plain C."""
    e = ctxs[0]
    n, t, nd, lo, hi = 64, 11, 9, 10, 17
    commits, shares = _round(e, n, t, nd, "plainc")
    shares[3 * n + 12, 5] ^= 1
    sh = _cols(shares, n, 0, nd, lo, hi)
    want = _reference(e, commits, t, 0, nd, lo, hi, sh)
    fx = tmp_path / "fx.bin"
    fx.write_bytes(np.array([n, t, nd, lo, hi], dtype=np.uint64).tobytes() + commits.tobytes() + sh.tobytes() + want.tobytes())
    exe = tmp_path / "dkg_columns_check"
    libdir = os.path.dirname(kb.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "dkg_columns_check.c"),
                           "-L", libdir, "-lkyber_b200", "-Wl,-rpath," + libdir, "-o", str(exe)])
    r = subprocess.run([str(exe), str(fx)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
