"""KB_ROUND_CHECK_BATCHED: DKG rounds checked as one random linear combination per dealer (dkgrlc.cuh).  Every case compares
the verdicts (and signature statuses) item by item with an EXACT context on the same inputs, samples against the oracle,
and asserts the number of dealers checked share by share."""
import hashlib
import importlib
import os
import subprocess

import numpy as np
import pytest

from helpers import ROOT, xof_bytes
from oracle import ed25519_bigint as O
from test_gpu_keyed_round import _sub, make_round

pytestmark = pytest.mark.gpu

L = O.L


@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


@pytest.fixture(scope="module")
def exact(kb):
    c = kb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def batched(kb):
    c = kb.Context(0)
    c.set_round_check("batched")
    yield c
    c.close()


def _torsion(order):
    """A point of the given order 2, 4 or 8 as an encoding."""
    t8 = O.point_decode(O.WEAK_KEYS[2])
    return O.point_encode(O._mul_int(8 // order, t8))


def _round(ctx, n, t, nd, tag):
    """Commitments and honest shares of nd dealers (random coefficients below 2^252)."""
    coeffs = np.frombuffer(xof_bytes(f"{tag}/coeffs", 32 * nd * t), dtype=np.uint8).reshape(nd * t, 32).copy()
    coeffs[:, 31] &= 0x0F
    commits = ctx.point_mul_base_batch(coeffs, 1).copy()
    shares = ctx.pripoly_eval_batch(coeffs, t, n).copy()
    return commits, shares


def _add_point(ctx, enc, p):
    return ctx.point_add_batch(enc.reshape(1, 32), np.frombuffer(p, dtype=np.uint8).reshape(1, 32))[0][0]


def _wrong_dealers(shares_ok, shares, n):
    return len({k // n for k in np.flatnonzero((shares_ok != shares).any(axis=1))})


def _compare(exact, batched, n, t, commits, shares, fallbacks, limbs=False):
    want = exact.dkg_verify_round(n, t, commits, shares, limbs=limbs)
    assert exact.round_fallbacks() == 0
    got = batched.dkg_verify_round(n, t, commits, shares, limbs=limbs)
    assert (got == want).all(), np.argwhere(got != want)[:10]
    assert batched.round_fallbacks() == fallbacks
    return got


def test_mode_argument_and_default(kb, exact):
    """A fresh context is EXACT (no fallback count), any mode other than 0 and 1 is KB_ERR_ARG, wipe keeps the mode."""
    c = kb.Context(0)
    try:
        assert c.round_fallbacks() == 0
        for bad in (2, -1, 7):
            assert c.L.kb_ctx_set_round_check(c.h, bad) == -1
        assert c.L.kb_ctx_set_round_check(None, 1) == -1
        n, t = 16, 3
        commits, shares = _round(c, n, t, 4, "rc/mode")
        shares[5, 3] ^= 1
        v0 = c.dkg_verify_round(n, t, commits, shares)
        assert c.round_fallbacks() == 0
        c.set_round_check("batched")
        c.wipe()
        assert (c.dkg_verify_round(n, t, commits, shares) == v0).all()
        assert c.round_fallbacks() == 1
        c.set_round_check("exact")
        assert (c.dkg_verify_round(n, t, commits, shares) == v0).all()
        assert c.round_fallbacks() == 0
    finally:
        c.close()


@pytest.mark.parametrize("wrong", [True, False])
def test_cfg4_shape_two_dealers(exact, batched, coracle, wrong):
    """n = 1024, t = 683 with dealer 1 carrying an order-8 point on C_1 (valid only where 8 | x).  With wrong shares both
    dealers fall back; without, both pass the combination and the torsion dealer gets the pattern 8 | x."""
    n, t, nd = 1024, 683, 2
    coeff = [[int.from_bytes(hashlib.sha512(b"rc-cfg4/%d/%d" % (d, j)).digest(), "little") % L for j in range(t)] for d in range(nd)]
    commits = exact.point_mul_base_batch(np.frombuffer(b"".join(c.to_bytes(32, "little") for row in coeff for c in row), dtype=np.uint8).reshape(-1, 32)).copy()
    shares = np.zeros((nd * n, 32), dtype=np.uint8)
    for d in range(nd):
        for i in range(n):
            v = 0
            for cj in reversed(coeff[d]):
                v = (v * (i + 1) + cj) % L
            shares[d * n + i] = np.frombuffer(v.to_bytes(32, "little"), dtype=np.uint8)
    want = np.ones((nd, n), dtype=np.uint8)
    if wrong:
        for d, i in ((0, 0), (0, 511), (0, 1023), (1, 7), (1, 640)):
            shares[d * n + i, 9] ^= 4
            want[d, i] = 0
    commits[t + 1] = _add_point(exact, commits[t + 1], O.WEAK_KEYS[2])
    torsion_ok = np.zeros(n, dtype=np.uint8)
    torsion_ok[7::8] = 1
    want[1] &= torsion_ok
    got = _compare(exact, batched, n, t, commits, shares, 2 if wrong else 0).reshape(nd, n)
    assert (got == want).all()
    for d, i in ((0, 0), (0, 1), (1, 7), (1, 8)):
        cs = commits[d * t:(d + 1) * t]
        assert coracle.vss_verify_deal([c.tobytes() for c in cs], i, shares[d * n + i].tobytes()) == int(got[d, i])


@pytest.mark.parametrize("t", [1, 2, 3, 4, 5, 43])
def test_torsion_positions_no_fallback(exact, batched, coracle, t):
    """Points of order 2, 4 and 8 on coefficients 0, 1, 2, 3 and t - 1, and even / odd pairs that cancel: honest shares, so
    no dealer falls back, and the verdicts are the exact ones for every residue of x mod 8."""
    n = 40
    cases = []
    for order in (2, 4, 8):
        for j in sorted({0, 1, 2, 3, t - 1}):
            if j < t:
                cases.append({j: _torsion(order)})
    t8, t8n = _torsion(8), O.point_encode(O.point_neg(O.point_decode(_torsion(8))))
    if t >= 3:
        cases.append({0: t8, 2: t8n})          # cancels for every x
        cases.append({1: _torsion(4), 2: _torsion(2)})
    if t >= 4:
        cases.append({1: t8, 3: t8n})          # cancels for odd x only
    cases.append({})
    nd = len(cases)
    commits, shares = _round(exact, n, t, nd, f"rc/torsion/{t}")
    for d, tdict in enumerate(cases):
        for j, p in tdict.items():
            commits[d * t + j] = _add_point(exact, commits[d * t + j], p)
    got = _compare(exact, batched, n, t, commits, shares, 0).reshape(nd, n)
    for d in (0, nd - 2):
        for i in (0, 1, 7):
            cs = [c.tobytes() for c in commits[d * t:(d + 1) * t]]
            assert coracle.vss_verify_deal(cs, i, shares[d * n + i].tobytes()) == int(got[d, i])


def test_bad_commitments(exact, batched, coracle):
    """Undecodable encodings and inconsistent limbs give 0 for the whole dealer, without a fallback."""
    n, t, nd = 24, 5, 9
    commits, shares = _round(exact, n, t, nd, "rc/bad")
    k = 0
    while coracle.point_decode_ok(bytes([k]) + b"\x13" * 31):
        k += 1
    enc = commits.copy()
    enc[2 * t + 1] = np.frombuffer(bytes([k]) + b"\x13" * 31, dtype=np.uint8)
    shares[7 * n + 3, 0] ^= 1
    got = _compare(exact, batched, n, t, enc, shares, 1).reshape(nd, n)
    assert not got[2].any() and got[0].all()
    limbs = np.stack([coracle.point_limbs(c.tobytes()) for c in commits])
    limbs[4 * t + 3, 7] += 1   # T Z != X Y
    got = _compare(exact, batched, n, t, limbs, shares, 1, limbs=True).reshape(nd, n)
    assert not got[4].any() and got[0].all()


def test_unreduced_and_high_shares(exact, batched):
    """Honest shares given as s + L (byte 31 <= 127) stay on the fast path; a share with byte 31 > 127 sends its dealer to
    the share-by-share check, whatever its verdict."""
    n, t, nd = 32, 7, 6
    commits, shares = _round(exact, n, t, nd, "rc/high")
    sl = shares.copy()
    for k in range(0, nd * n, 3):
        v = int.from_bytes(sl[k].tobytes(), "little") + L
        sl[k] = np.frombuffer(v.to_bytes(32, "little"), dtype=np.uint8)
    _compare(exact, batched, n, t, commits, sl, 0)
    hi = shares.copy()
    for k, m in ((1 * n + 4, 8), (3 * n + 9, 9), (3 * n + 10, 15)):
        v = int.from_bytes(hi[k].tobytes(), "little") + m * L
        hi[k] = np.frombuffer((v % (1 << 256)).to_bytes(32, "little"), dtype=np.uint8)
        assert hi[k, 31] > 127
    _compare(exact, batched, n, t, commits, hi, 2)


@pytest.mark.parametrize("kind", ["none", "one-per-dealer", "0.1%", "all"])
def test_wrong_share_fractions(exact, batched, kind):
    """The fallback count is the number of dealers that have a wrong share."""
    n, t, nd = 128, 43, 256
    commits, shares = _round(exact, n, t, nd, "rc/frac")
    bad = shares.copy()
    rng = np.random.default_rng(11)
    if kind == "one-per-dealer":
        idx = np.arange(nd) * n + rng.integers(0, n, nd)
    elif kind == "0.1%":
        idx = rng.choice(nd * n, (nd * n) // 1000, replace=False)
    elif kind == "all":
        idx = np.arange(nd * n)
    else:
        idx = np.zeros(0, dtype=np.int64)
    bad[idx, 5] ^= 0x20
    _compare(exact, batched, n, t, commits, bad, _wrong_dealers(shares, bad, n))


def test_process_round_keyed_and_unkeyed(exact, batched, coracle):
    """kb_dkg_process_round and kb_dkg_process_round_keyed on the fixtures of the keyed-round tests: verdicts and both
    signature statuses as on an EXACT context."""
    n, t, nd = 20, 7, 37
    R = make_round(exact, coracle, n, t, nd, "rc/keyed")
    wrong = len({k // n for k in (0, (nd * n) // 2, nd * n - 1)})
    ke, kbt = exact.keyset(R["dkeys"]), batched.keyset(R["dkeys"])
    try:
        want = exact.dkg_process_round_keyed(n, t, R["commits"], R["shares"], ke, deal=R["deal"], resp=R["resp"])
        got = batched.dkg_process_round_keyed(n, t, R["commits"], R["shares"], kbt, deal=R["deal"], resp=R["resp"])
        assert batched.round_fallbacks() == wrong
        for a, b in zip(want, got):
            assert (a == b).all()
        assert (got[0] == R["want_v"]).all()
        k = np.arange(nd * n)
        deal = (R["dkeys"][k // n],) + tuple(R["deal"])
        resp = (R["vkeys"][k % n],) + tuple(R["resp"])
        want = exact.dkg_process_round(n, t, R["commits"], R["shares"], deal=deal, resp=resp)
        got = batched.dkg_process_round(n, t, R["commits"], R["shares"], deal=deal, resp=resp)
        assert batched.round_fallbacks() == wrong
        for a, b in zip(want, got):
            assert (a == b).all()
    finally:
        ke.close()
        kbt.close()


def test_device_form_on_a_stream(exact, batched):
    """kb_dev_dkg_verify_round[_limbs] on a side stream: same verdicts, the fallback count waits for that stream."""
    import torch

    n, t, nd = 64, 11, 40
    commits, shares = _round(exact, n, t, nd, "rc/dev")
    shares[3 * n + 2, 4] ^= 1
    shares[39 * n + 63, 4] ^= 1
    want = exact.dkg_verify_round(n, t, commits, shares)
    dev = torch.device("cuda", 0)
    d_c, d_s = torch.from_numpy(commits).to(dev), torch.from_numpy(shares).to(dev)
    d_v = torch.full((nd * n,), 99, dtype=torch.uint8, device=dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        batched.dev_dkg_verify_round(n, t, nd, d_c, d_s, d_v)
    assert batched.round_fallbacks() == 2
    side.synchronize()
    assert (d_v.cpu().numpy() == want).all()


@pytest.fixture(scope="module", params=["one", "all"])
def mctx(kb, request):
    import torch

    ngpu = torch.cuda.device_count()
    if request.param == "all" and ngpu < 2:
        pytest.skip("a single GPU is visible")
    m = kb.MultiContext([0] if request.param == "one" else list(range(min(ngpu, 8))))
    yield m
    m.close()


def test_multi_device_round(kb, exact, mctx, coracle):
    """MultiContext.set_round_check applies to every device: the split round gives the exact verdicts and statuses, and the
    per-device fallback counts add up to the dealers with a wrong share."""
    n, t, nd = 20, 7, 37
    R = make_round(exact, coracle, n, t, nd, "rc/mctx")
    wrong = len({k // n for k in (0, (nd * n) // 2, nd * n - 1)})
    mctx.set_round_check("batched")
    mk, ke = mctx.keyset(R["dkeys"]), exact.keyset(R["dkeys"])
    try:
        want = exact.dkg_process_round_keyed(n, t, R["commits"], R["shares"], ke, deal=R["deal"], resp=R["resp"])
        got = mctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], mk, deal=R["deal"], resp=R["resp"])
        for a, b in zip(want, got):
            assert (a == b).all()
        assert (mctx.dkg_verify_round(n, t, R["commits"], R["shares"]) == want[0]).all()
        import ctypes

        total = 0
        for k in range(len(mctx.devices)):
            v = ctypes.c_uint64()
            assert mctx.L.kb_ctx_round_fallbacks(mctx.L.kb_mctx_ctx(mctx.h, k), ctypes.byref(v)) == 0
            total += v.value
        assert total == wrong
    finally:
        mk.close()
        ke.close()
        mctx.set_round_check("exact")


def test_round_batched_from_plain_c(kb, exact, tmp_path):
    """tests/c/round_batched_check.c: the mode, the fallback count and the verdicts from plain C (gcc, -lkyber_b200)."""
    n, t, nd = 48, 9, 21
    commits, shares = _round(exact, n, t, nd, "rc/c")
    ok = shares.copy()
    for k in (5, 6, 17 * n + 40):
        shares[k, 2] ^= 8
    want = exact.dkg_verify_round(n, t, commits, shares)
    fx = tmp_path / "fixture.bin"
    with open(fx, "wb") as f:
        f.write(np.array([n, t, nd, _wrong_dealers(ok, shares, n)], dtype=np.uint64).tobytes())
        for a in (commits, shares, want):
            f.write(np.ascontiguousarray(a).tobytes())
    exe = tmp_path / "round_batched_check"
    libdir = os.path.dirname(kb.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "round_batched_check.c"),
                           "-L", libdir, "-lkyber_b200", "-Wl,-rpath," + libdir, "-o", str(exe)])
    r = subprocess.run([str(exe), str(fx)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "mismatches=0" in r.stdout
