"""Keyed DKG rounds (kb_dkg_process_round_keyed / kb_dev_dkg_process_round_keyed) and key sets on the multi-device
context (kb_mctx_keyset_*, kb_mctx_dkg_process_round_keyed): item for item what the unkeyed round and the general
verifiers (and the C oracle) return for the same keys."""
import importlib
import os
import subprocess

import numpy as np
import pytest

from helpers import ROOT, make_sig_batch, pack_batch, xof_bytes

pytestmark = pytest.mark.gpu

NONCANON_ID = bytes([0xEE]) + b"\xff" * 30 + b"\x7f"    # y = p + 1 = 1: the identity, non-canonically encoded
SMALL_ORDER = bytes([0x01]) + b"\x00" * 31               # the identity


@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


@pytest.fixture(scope="module")
def ctx(kb):
    c = kb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module", params=["one", "all"])
def mctx(kb, request):
    import torch

    ngpu = torch.cuda.device_count()
    if request.param == "all" and ngpu < 2:
        pytest.skip("a single GPU is visible")
    m = kb.MultiContext([0] if request.param == "one" else list(range(min(ngpu, 8))))
    yield m
    m.close()


def _undecodable(coracle) -> bytes:
    k = 0
    while coracle.point_decode_ok(bytes([k]) + b"\x13" * 31):
        k += 1
    return bytes([k]) + b"\x13" * 31


def _signed(ctx, seeds, signer, mlen, tag, rng):
    """(flat, off, sig) of len(signer) messages of mlen bytes, message k signed by seeds[signer[k]]; every 8th item is
    damaged in s, R or the message, in turn."""
    m = signer.shape[0]
    flat = np.frombuffer(xof_bytes(tag, mlen * m), dtype=np.uint8).copy()
    off = np.arange(m + 1, dtype=np.uint64) * np.uint64(mlen)
    sig, _ = ctx.eddsa_sign_batch(seeds[signer], flat, off)
    sig = sig.copy()
    for k in range(3, m, 8):
        kind = (k // 8) % 3
        if kind == 0:
            sig[k, 32 + rng.integers(0, 31)] ^= 1 << rng.integers(0, 8)
        elif kind == 1:
            sig[k, rng.integers(0, 32)] ^= 1 << rng.integers(0, 8)
        else:
            flat[mlen * k + rng.integers(0, mlen)] ^= 1
    return flat, off, sig


def _keys(ctx, seeds):
    z = np.zeros((seeds.shape[0], 0), dtype=np.uint8)
    _, pk = ctx.eddsa_sign_batch(seeds, z.reshape(-1), np.zeros(seeds.shape[0] + 1, dtype=np.uint64))
    return pk.copy()


def make_round(ctx, coracle, n, t, nd, tag, nverifier_keys=None, bad_keys=True):
    """A round of nd dealers and n verifiers: commitments, shares (three damaged), deal messages of 128 bytes signed by
    their dealer and responses of 32 bytes signed by their verifier.  The dealer and verifier keys are one participant set
    unless nverifier_keys is given.  With bad_keys, three participants' keys are replaced by a non-canonical, a
    small-order and an undecodable encoding (their signatures stay those of the original keys)."""
    rng = np.random.default_rng(int.from_bytes(xof_bytes(f"{tag}/rng", 8), "little"))
    coeffs = np.frombuffer(xof_bytes(f"{tag}/coeffs", 32 * nd * t), dtype=np.uint8).reshape(nd * t, 32).copy()
    coeffs[:, 31] &= 0x0F
    commits = ctx.point_mul_base_batch(coeffs, 1)
    shares = ctx.pripoly_eval_batch(coeffs, t, n).copy()
    want_v = np.ones(nd * n, dtype=np.uint8)
    for k in (0, (nd * n) // 2, nd * n - 1):
        shares[k, 1] ^= 4
        want_v[k] = 0
    m = nd * n
    nkeys = max(nd, n)
    dseeds = np.frombuffer(xof_bytes(f"{tag}/dealers", 32 * nkeys), dtype=np.uint8).reshape(nkeys, 32)
    vseeds = dseeds if nverifier_keys is None else np.frombuffer(xof_bytes(f"{tag}/verifiers", 32 * nverifier_keys), dtype=np.uint8).reshape(nverifier_keys, 32)
    k = np.arange(m)
    deal = _signed(ctx, dseeds, k // n, 128, f"{tag}/deal", rng)
    resp = _signed(ctx, vseeds, k % n, 32, f"{tag}/resp", rng)
    dkeys = _keys(ctx, dseeds)
    vkeys = dkeys if nverifier_keys is None else _keys(ctx, vseeds)
    if bad_keys:
        for i, enc in ((1, NONCANON_ID), (min(4, n - 1), SMALL_ORDER), (min(6, n - 1), _undecodable(coracle))):
            dkeys[i] = np.frombuffer(enc, dtype=np.uint8)
            vkeys[i] = dkeys[i]
    return dict(n=n, t=t, nd=nd, commits=commits, shares=shares, want_v=want_v, deal=deal, resp=resp, dkeys=dkeys, vkeys=vkeys)


def _pk_batch(keys, signer, batch):
    return (keys[signer],) + tuple(batch)


def _unkeyed(ctx, R, lo=0, hi=None):
    hi = R["nd"] if hi is None else hi
    n = R["n"]
    k = np.arange(lo * n, hi * n)
    deal = _sub(R["deal"], lo * n, hi * n)
    resp = _sub(R["resp"], lo * n, hi * n)
    return ctx.dkg_process_round(n, R["t"], R["commits"], R["shares"], deal=_pk_batch(R["dkeys"], k // n, deal), resp=_pk_batch(R["vkeys"], k % n, resp), dealer_lo=lo, dealer_hi=hi)


def _sub(batch, a, b):
    """items [a, b) of (flat, off, sig) with rebased offsets"""
    flat, off, sig = batch
    return flat[int(off[a]):int(off[b])], off[a:b + 1] - off[a], sig[a:b]


@pytest.mark.parametrize("n,t,nd", [(20, 7, 37), (256, 171, 24)])
def test_keyed_round_matches_unkeyed_and_oracle(ctx, coracle, n, t, nd):
    R = make_round(ctx, coracle, n, t, nd, f"keyed/{n}")
    m = nd * n
    k = np.arange(m)
    v0, d0, r0 = _unkeyed(ctx, R)
    assert (v0 == R["want_v"]).all()
    assert (d0 == coracle.verify_batch(*_pk_batch(R["dkeys"], k // n, R["deal"]), nthreads=8, schnorr=True)).all()
    assert (r0 == coracle.verify_batch(*_pk_batch(R["vkeys"], k % n, R["resp"]), nthreads=8, schnorr=True)).all()
    for st in (d0, r0):
        assert {0, 8} <= set(st.tolist()) and {5, 6, 7} & set(st.tolist())   # damaged signatures and keys are both met
    ks = ctx.keyset(R["dkeys"])
    try:
        v, d, r = ctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], ks, deal=R["deal"], resp=R["resp"])
        assert (v == v0).all()
        assert (d == d0).all(), np.nonzero(d != d0)[0][:10]
        assert (r == r0).all(), np.nonzero(r != r0)[0][:10]
    finally:
        ks.close()


def test_keyed_round_ranges_limbs_and_single_batches(ctx, coracle):
    """A dealer sub-range with absolute dealer keys (offsets absolute into the whole message array, and rebased), the
    limbs form, deal-only and response-only calls."""
    n, t, nd = 20, 7, 37
    R = make_round(ctx, coracle, n, t, nd, "keyed/ranges")
    v0, d0, r0 = _unkeyed(ctx, R)
    ks = ctx.keyset(R["dkeys"])
    try:
        lo, hi = 8, 21
        a, b = lo * n, hi * n
        absolute = lambda batch: (batch[0], batch[1][a:b + 1], batch[2][a:b])
        for cut in (absolute, lambda batch: _sub(batch, a, b)):
            v, d, r = ctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], ks, deal=cut(R["deal"]), resp=cut(R["resp"]), dealer_lo=lo, dealer_hi=hi)
            assert (v[a:b] == v0[a:b]).all() and (d == d0[a:b]).all() and (r == r0[a:b]).all()
        vs, ds, rs = _unkeyed(ctx, R, lo, hi)
        assert (ds == d0[a:b]).all() and (rs == r0[a:b]).all()
        limbs = np.stack([coracle.point_limbs(c.tobytes()) for c in R["commits"]])
        v, d, r = ctx.dkg_process_round_keyed(n, t, limbs, R["shares"], ks, deal=R["deal"], resp=R["resp"], limbs=True)
        assert (v == v0).all() and (d == d0).all() and (r == r0).all()
        v, d, r = ctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], ks, deal=R["deal"])
        assert (v == v0).all() and (d == d0).all() and r is None
        v, d, r = ctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], ks, resp=R["resp"])
        assert (v == v0).all() and d is None and (r == r0).all()
    finally:
        ks.close()


def test_keyed_round_separate_dealer_and_verifier_sets(ctx, coracle):
    """Resharing: 13 dealers (old nodes) and 20 verifiers (new nodes) with key sets of their own."""
    n, t, nd = 20, 7, 13
    R = make_round(ctx, coracle, n, t, nd, "keyed/reshare", nverifier_keys=n)
    R["dkeys"] = R["dkeys"][:nd].copy()
    v0, d0, r0 = _unkeyed(ctx, R)
    k = np.arange(nd * n)
    assert (r0 == coracle.verify_batch(*_pk_batch(R["vkeys"], k % n, R["resp"]), nthreads=8, schnorr=True)).all()
    kd, kv = ctx.keyset(R["dkeys"]), ctx.keyset(R["vkeys"])
    try:
        v, d, r = ctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], kd, kv, deal=R["deal"], resp=R["resp"])
        assert (v == v0).all() and (d == d0).all() and (r == r0).all()
    finally:
        kd.close()
        kv.close()


def _to_dev(*arrays):
    import torch

    dev = torch.device("cuda", 0)
    return [torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else np.ascontiguousarray(a)).to(dev) for a in arrays]


def test_keyed_round_device_form(ctx, coracle):
    """kb_dev_dkg_process_round_keyed on a non-default stream gives what the host form gives, for the whole round and for
    a dealer sub-range whose arrays start at its first dealer."""
    import torch

    n, t, nd = 20, 7, 37
    R = make_round(ctx, coracle, n, t, nd, "keyed/dev")
    ks = ctx.keyset(R["dkeys"])
    side = torch.cuda.Stream()
    try:
        hv, hd, hr = ctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], ks, deal=R["deal"], resp=R["resp"])
        for lo, hi in ((0, nd), (8, 21)):
            a, b = lo * n, hi * n
            deal, resp = _sub(R["deal"], a, b), _sub(R["resp"], a, b)
            d_c, d_s = _to_dev(R["commits"][lo * t:hi * t], R["shares"][a:b])
            d_deal, d_resp = _to_dev(*deal), _to_dev(*resp)
            d_v, d_ds, d_rs = (torch.full((b - a,), 99, dtype=torch.uint8, device="cuda") for _ in range(3))
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                ctx.dev_dkg_process_round_keyed(n, t, hi - lo, d_c, d_s, d_v, ks, deal=(*d_deal, d_ds), resp=(*d_resp, d_rs), dealer_lo=lo)
            side.synchronize()
            assert (d_v.cpu().numpy() == hv[a:b]).all()
            assert (d_ds.cpu().numpy() == hd[a:b]).all() and (d_rs.cpu().numpy() == hr[a:b]).all()
    finally:
        ks.close()


def test_keyed_round_argument_errors(kb, ctx, coracle):
    """Every refusal of the keyed round is KB_ERR_ARG before anything is launched."""
    import torch

    n, t, nd = 20, 7, 37
    R = make_round(ctx, coracle, n, t, nd, "keyed/errors", bad_keys=False)
    ks = ctx.keyset(R["dkeys"])
    short = ctx.keyset(R["dkeys"][:nd - 1])
    few = ctx.keyset(R["dkeys"][:n - 1])
    other_ctx = kb.Context(0)
    other = other_ctx.keyset(R["dkeys"])
    args = (n, t, R["commits"], R["shares"])
    try:
        before = ctx.launches
        cases = [
            dict(dealers=short, verifiers=ks, deal=R["deal"]),                     # dealers->nkeys < dealer_hi
            dict(dealers=short, verifiers=ks, resp=R["resp"]),                     # ... whether or not the deals are given
            dict(dealers=ks, verifiers=few, resp=R["resp"]),                       # verifiers->nkeys < n
            dict(dealers=other, verifiers=ks, deal=R["deal"]),                     # a key set of another context
            dict(dealers=ks, verifiers=other, resp=R["resp"]),
            dict(dealers=None, verifiers=ks, deal=R["deal"]),                      # deals without a dealer key set
            dict(dealers=None, verifiers=None, resp=R["resp"]),                    # responses without a verifier key set
        ]
        for c in cases:
            with pytest.raises(kb.KBError, match="-1"):
                ctx.dkg_process_round_keyed(*args, c.pop("dealers"), **c)
        # a dealer range beyond the key set
        with pytest.raises(kb.KBError, match="-1"):
            ctx.dkg_process_round_keyed(*args, short, deal=_sub(R["deal"], 30 * n, nd * n), dealer_lo=30, dealer_hi=nd)
        d_c, d_s = _to_dev(R["commits"], R["shares"])
        d_deal = _to_dev(*R["deal"])
        d_v, d_st = (torch.zeros(nd * n, dtype=torch.uint8, device="cuda") for _ in range(2))
        for dealers, lo, nd_ in ((short, 0, nd), (ks, 1, nd), (other, 0, nd), (None, 0, nd)):
            with pytest.raises(kb.KBError, match="-1"):
                ctx.dev_dkg_process_round_keyed(n, t, nd_, d_c, d_s, d_v, dealers, ks, deal=(*d_deal, d_st), dealer_lo=lo)
        torch.cuda.synchronize()
        assert ctx.launches == before
        # still usable
        v0, d0, _ = _unkeyed(ctx, R)
        v, d, _ = ctx.dkg_process_round_keyed(*args, ks, deal=R["deal"])
        assert (v == v0).all() and (d == d0).all()
        v, d, _ = ctx.dkg_process_round_keyed(*args, short, deal=_sub(R["deal"], 0, 36 * n), dealer_hi=36)
        assert (d == d0[:36 * n]).all()
    finally:
        other.close()
        other_ctx.close()
        for x in (ks, short, few):
            x.close()


def test_mctx_keyset_verify_matches_keyset(kb, ctx, mctx, golden_records):
    """MultiKeySet.verify_batch split by index: what the single-context KeySet returns, at 1003 items (uneven shards) and
    at 1; an index outside the set is refused before any device starts."""
    for nitems in (1003, 1):
        pks, msgs, sigs = make_sig_batch(golden_records[:300], nitems, bad_every=4)
        pk, flat, off, sg = pack_batch(pks, msgs, sigs)
        keys, inv = np.unique(pk, axis=0, return_inverse=True)
        key_idx = inv.reshape(-1).astype(np.uint32)
        ks, mk = ctx.keyset(keys), mctx.keyset(keys)
        try:
            for schnorr in (False, True):
                want = ks.verify_batch(key_idx, flat, off, sg, schnorr=schnorr)
                assert (want == ctx.verify_batch(pk, flat, off, sg, schnorr=schnorr)).all()
                assert (mk.verify_batch(key_idx, flat, off, sg, schnorr=schnorr) == want).all()
            before = mctx.launches
            bad = key_idx.copy()
            bad[-1] = keys.shape[0]
            with pytest.raises(kb.KBError, match="-1"):
                mk.verify_batch(bad, flat, off, sg)
            assert mctx.launches == before
        finally:
            ks.close()
            mk.close()


def test_mctx_keyed_round_matches_single_device(kb, ctx, mctx, coracle):
    """The keyed round split by dealer: verdicts and statuses equal the single-device keyed round's, with one key set for
    both roles and with separate dealer and verifier sets."""
    n, t, nd = 20, 7, 37
    R = make_round(ctx, coracle, n, t, nd, "keyed/mctx")
    ks = ctx.keyset(R["dkeys"])
    mk = mctx.keyset(R["dkeys"])
    mv = mctx.keyset(R["vkeys"][:n])
    try:
        v0, d0, r0 = ctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], ks, deal=R["deal"], resp=R["resp"])
        v, d, r = mctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], mk, deal=R["deal"], resp=R["resp"])
        assert (v == v0).all() and (d == d0).all() and (r == r0).all()
        v, d, r = mctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], mk, mv, deal=R["deal"], resp=R["resp"])
        assert (v == v0).all() and (d == d0).all() and (r == r0).all()
        v, d, r = mctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], mk, resp=R["resp"])
        assert (v == v0).all() and d is None and (r == r0).all()
        before = mctx.launches
        with pytest.raises(kb.KBError, match="-1"):
            mctx.dkg_process_round_keyed(n, t, R["commits"], R["shares"], mv, deal=R["deal"])   # 20 keys, 37 dealers
        assert mctx.launches == before
    finally:
        ks.close()
        mk.close()
        mv.close()


def test_keyed_round_from_plain_c(kb, ctx, coracle, tmp_path):
    """tests/c/keyed_round_check.c: the keyed round, the multi-device key set and the multi-device keyed round from plain
    C (gcc, -lkyber_b200), on a fixture whose expected bytes come from the oracle."""
    n, t, nd = 20, 7, 37
    R = make_round(ctx, coracle, n, t, nd, "keyed/c")
    m = nd * n
    k = np.arange(m)
    want_d = coracle.verify_batch(*_pk_batch(R["dkeys"], k // n, R["deal"]), nthreads=8, schnorr=True).astype(np.uint8)
    want_r = coracle.verify_batch(*_pk_batch(R["vkeys"], k % n, R["resp"]), nthreads=8, schnorr=True).astype(np.uint8)
    fx = tmp_path / "fixture.bin"
    with open(fx, "wb") as f:
        f.write(np.array([n, t, nd, R["dkeys"].shape[0], R["deal"][0].size, R["resp"][0].size], dtype=np.uint64).tobytes())
        for a in (R["dkeys"], R["commits"], R["shares"], R["deal"][2], R["deal"][1], R["deal"][0], R["resp"][2], R["resp"][1], R["resp"][0], R["want_v"], want_d, want_r):
            f.write(np.ascontiguousarray(a).tobytes())
    exe = tmp_path / "keyed_round_check"
    libdir = os.path.dirname(kb.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "keyed_round_check.c"),
                           "-L", libdir, "-lkyber_b200", "-Wl,-rpath," + libdir, "-o", str(exe)])
    r = subprocess.run([str(exe), str(fx)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "mismatches=0" in r.stdout
