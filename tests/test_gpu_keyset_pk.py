"""Key sets by public-key bytes on the B200: kb_keyset_verify_pk_batch / kb_dev_keyset_verify_pk /
kb_mctx_keyset_verify_pk_batch return, item for item, what kb_eddsa_verify_batch / kb_schnorr_verify_batch (and the C
oracle) return on the same inputs, and count as hits exactly the items whose 32 pk bytes are registered."""
import ctypes
import importlib
import os
import sys

import numpy as np
import pytest

from helpers import NONCANONICAL, ROOT, WEAK_KEYS, _off_curve, make_mixed_order_sigs, make_sig_batch, pack_batch

sys.path.insert(0, ROOT)
import bench  # noqa: E402

pytestmark = pytest.mark.gpu

BIG = (1 << 20) + 37
SMALL = (1, 7, 8, 9)
KEYS = (1, 7, 1024, 65536)
FRACS = ((0, 1), (1, 2), (63, 64), (1, 1))
KB_OK, KB_ERR_ARG = 0, -1


@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


@pytest.fixture(scope="module")
def ctx(kb):
    c = kb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def mctx(kb):
    m = kb.MultiContext([0])
    yield m
    m.close()


def _scalars(tag, n):
    a = bench.xof(tag, 32 * n).reshape(n, 32).copy()
    a[:, 31] &= 0x0F
    return a


@pytest.fixture(scope="module")
def registered(ctx, mctx):
    """Per K: (secret scalars, keys, KeySet, MultiKeySet), built once for the module."""
    sets = {}
    for k in KEYS:
        a = _scalars(f"kyber-b200/test/keyset_pk/keys/{k}", k)
        keys = ctx.point_mul_base_batch(a)
        sets[k] = (a, keys, ctx.keyset(keys), mctx.keyset(keys))
    yield sets
    for _, _, ks, mks in sets.values():
        ks.close()
        mks.close()


def _rows(a):
    a = np.ascontiguousarray(a)
    return a.view(np.dtype((np.void, a.shape[1]))).reshape(-1)


def _host_hits(pk, keys):
    return int(np.isin(_rows(pk), _rows(keys)).sum())


def _make_batch(ctx, a_reg, keys, n, frac, seed):
    """n signatures over 64-byte messages: round(frac n) of them under registered keys (random positions and keys), the
    rest under 4096 other keys; then every 64th item spoiled in bench.spoil's nine classes (three of which replace pk)."""
    rng = np.random.default_rng(seed)
    k = keys.shape[0]
    a_un = _scalars(f"kyber-b200/test/keyset_pk/others/{seed}", 4096)
    keys_un = ctx.point_mul_base_batch(a_un)
    hit = np.zeros(n, dtype=bool)
    hit[rng.permutation(n)[: round(n * frac[0] / frac[1])]] = True
    ki = rng.integers(0, k, size=n)
    ku = rng.integers(0, 4096, size=n)
    a = np.where(hit[:, None], a_reg[ki], a_un[ku])
    pk = np.where(hit[:, None], keys[ki], keys_un[ku])
    r = _scalars(f"kyber-b200/test/keyset_pk/nonces/{seed}", n)
    msg = bench.xof(f"kyber-b200/test/keyset_pk/msgs/{seed}", 64 * n).copy()
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(64)
    R = ctx.point_mul_base_batch(r)
    s = ctx.sc_muladd_batch(ctx.challenge_batch(R, pk, msg, off), a, r)
    sig = np.concatenate([R, s], axis=1)
    bench.spoil(pk, msg, sig, 0, n)
    return pk, msg, off, sig


def _to_dev(dev, *arrays):
    import torch

    out = []
    for a in arrays:
        if a.dtype == np.uint64:
            a = a.view(np.int64)
        out.append(torch.from_numpy(a if a.size else np.zeros(1, dtype=a.dtype)).to(dev))
    return out


def _dev_verify_pk(ks, pk, flat, off, sg, schnorr, stream=None):
    """(statuses, hits) of kb_dev_keyset_verify_pk, on `stream` (or torch's current one)."""
    import torch

    dev = torch.device("cuda", 0)
    n = pk.shape[0]
    d_pk, d_msg, d_off, d_sig = _to_dev(dev, pk, flat, off, sg)
    d_st = torch.full((max(n, 1),), 99, dtype=torch.uint8, device=dev)
    d_hits = torch.full((1,), -1, dtype=torch.int64, device=dev)
    s = stream if stream is not None else torch.cuda.current_stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ks.dev_verify_pk(n, d_pk, d_msg, d_off, d_sig, d_st, schnorr=schnorr, hits=d_hits)
    s.synchronize()
    return d_st.cpu().numpy()[:n], int(d_hits.cpu()[0])


def _check_all_forms(ctx, keys, ks, mks, pk, flat, off, sg, schnorr, want=None):
    """Every form against the general verifier (or `want`), and the hit count against the host's."""
    if want is None:
        want = ctx.verify_batch(pk, flat, off, sg, schnorr=schnorr)
    hits = _host_hits(pk, keys)
    got, h = ks.verify_pk_batch(pk, flat, off, sg, schnorr=schnorr, return_hits=True)
    assert (got == want).all(), np.nonzero(got != want)[0][:10]
    assert h == hits
    got, h = _dev_verify_pk(ks, pk, flat, off, sg, schnorr)
    assert (got == want).all(), np.nonzero(got != want)[0][:10]
    assert h == hits
    got, h = mks.verify_pk_batch(pk, flat, off, sg, schnorr=schnorr, return_hits=True)
    assert (got == want).all(), np.nonzero(got != want)[0][:10]
    assert h == hits
    return want, hits


@pytest.mark.parametrize("frac", FRACS, ids=lambda f: f"{f[0]}of{f[1]}")
@pytest.mark.parametrize("nkeys", KEYS)
def test_pk_grid(ctx, coracle, registered, nkeys, frac):
    """2^20 + 37 items at the hit fraction, and its first 1, 7, 8 and 9 items, in all three forms and both schemes."""
    a_reg, keys, ks, mks = registered[nkeys]
    pk, flat, off, sg = _make_batch(ctx, a_reg, keys, BIG, frac, seed=nkeys * 101 + frac[0])
    for schnorr in (False, True):
        want, hits = _check_all_forms(ctx, keys, ks, mks, pk, flat, off, sg, schnorr)
        if frac == (0, 1):
            assert hits == 0
        elif frac == (1, 1):   # bench.spoil replaces pk (by unregistered bytes) in three classes of nine
            assert hits == BIG - sum(1 for i in range(63, BIG, 64) if (i // 64) % 9 in (4, 5, 8))
        m = 2048
        assert (want[:m] == coracle.verify_batch(pk[:m], flat[: 64 * m], off[: m + 1], sg[:m], nthreads=8, schnorr=schnorr)).all()
        for n in SMALL:
            # a batch that may be all hits, all misses or one of each, and not a multiple of 8 for the compression
            _check_all_forms(ctx, keys, ks, mks, pk[:n], flat[: 64 * n], off[: n + 1], sg[:n], schnorr, want=want[:n])


def _special_batch(golden_records):
    """Registered keys that are small-order, not canonical, undecodable or repeated, the same points under other
    encodings (not registered), and signatures under the golden keys (half registered) and under mixed-order keys."""
    ident_sign = bytes([1]) + bytes(30) + bytes([0x80])      # x = 0 with the sign bit set
    ident_plus_p = bytes([0xEE]) + b"\xff" * 30 + b"\x7f"    # y = 1 + p
    minus1_sign = bytes([0xEC]) + b"\xff" * 30 + b"\xff"     # y = -1 (order 2) with the sign bit set
    good, bad = make_mixed_order_sigs(24, seed=5)
    pks, msgs, sigs = make_sig_batch(golden_records, 2000, bad_every=2)
    pks += [x[0] for x in good + bad]
    msgs += [x[1] for x in good + bad]
    sigs += [x[2] for x in good + bad]
    special = [WEAK_KEYS[1], WEAK_KEYS[0], WEAK_KEYS[2], WEAK_KEYS[4], NONCANONICAL, _off_curve(7)]   # identity, 0, order 8, order 2, ...
    others = [ident_sign, ident_plus_p, minus1_sign]
    for i, p in enumerate(special + others):
        for j in range(5):
            rec = golden_records[(17 * i + j) % len(golden_records)]
            pks.append(p)
            msgs.append(rec[3])
            sigs.append(rec[2] if j % 2 else WEAK_KEYS[1] + rec[2][32:])
    pk, flat, off, sg = pack_batch(pks, msgs, sigs)
    distinct = np.unique(pk, axis=0)
    normal = distinct[~np.isin(_rows(distinct), _rows(np.frombuffer(b"".join(special + others), dtype=np.uint8).reshape(-1, 32)))]
    reg = np.concatenate([np.frombuffer(b"".join(special), dtype=np.uint8).reshape(-1, 32), normal[::2], normal[:3], normal[::2][:5]])
    return pk, flat, off, sg, reg, others


@pytest.mark.parametrize("schnorr", [False, True])
def test_pk_special_keys_and_duplicates(ctx, mctx, coracle, golden_records, schnorr):
    """Golden records with every mutation class (lengths 0 .. 1023), mixed-order keys, registered keys that are
    small-order, non-canonical or undecodable (hits), other encodings of registered points (misses), duplicate keys."""
    pk, flat, off, sg, reg, others = _special_batch(golden_records)
    want = coracle.verify_batch(pk, flat, off, sg, nthreads=8, schnorr=schnorr)
    assert (ctx.verify_batch(pk, flat, off, sg, schnorr=schnorr) == want).all()
    ks, mks = ctx.keyset(reg), mctx.keyset(reg)
    try:
        _, hits = _check_all_forms(ctx, reg, ks, mks, pk, flat, off, sg, schnorr, want=want)
        other_rows = _rows(np.frombuffer(b"".join(others), dtype=np.uint8).reshape(-1, 32))
        assert not np.isin(other_rows, _rows(reg)).any()
        assert 0 < hits < pk.shape[0]
    finally:
        ks.close()
        mks.close()


def test_pk_lookup_bounds_and_seeds(ctx, registered):
    """2^20 random pks that are not registered all miss in a set of 65 536 keys; two sets built from the same keys (with
    their own seeds) give the same statuses and hits."""
    import torch

    _, keys, ks, _ = registered[65536]
    n = 1 << 20
    pk = bench.xof("kyber-b200/test/keyset_pk/strangers", 32 * n).reshape(n, 32).copy()
    assert not np.isin(_rows(pk), _rows(keys)).any()
    sg = bench.xof("kyber-b200/test/keyset_pk/stranger_sigs", 64 * n).reshape(n, 64).copy()
    flat = bench.xof("kyber-b200/test/keyset_pk/stranger_msgs", 16 * n).copy()
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(16)
    want = ctx.verify_batch(pk, flat, off, sg)
    got, h = _dev_verify_pk(ks, pk, flat, off, sg, False)
    assert h == 0 and (got == want).all()
    # same keys, two sets: a mixed batch
    a_reg, keys1k, _, _ = registered[1024]
    bpk, bflat, boff, bsg = _make_batch(ctx, a_reg, keys1k, 50000, (1, 2), seed=99)
    s1, s2 = ctx.keyset(keys1k), ctx.keyset(keys1k)
    try:
        r1 = s1.verify_pk_batch(bpk, bflat, boff, bsg, schnorr=True, return_hits=True)
        r2 = s2.verify_pk_batch(bpk, bflat, boff, bsg, schnorr=True, return_hits=True)
        assert r1[1] == r2[1] == _host_hits(bpk, keys1k)
        assert (r1[0] == r2[0]).all() and (r1[0] == ctx.verify_batch(bpk, bflat, boff, bsg, schnorr=True)).all()
    finally:
        s1.close()
        s2.close()
    torch.cuda.synchronize()


def test_pk_streams_scratch_wipe_destroy(ctx, registered, golden_records):
    """The device form on a side stream between kb_dev_eddsa_verify and kb_dev_keyset_verify on two other streams of the
    same context; growth of the scratch from a small batch to a large one; kb_ctx_wipe between calls; destroy after use."""
    import torch

    dev = torch.device("cuda", 0)
    a_reg, keys, _, _ = registered[7]
    ks = ctx.keyset(keys)
    small = _make_batch(ctx, a_reg, keys, 100, (1, 2), seed=3)
    large = _make_batch(ctx, a_reg, keys, 300000, (63, 64), seed=4)
    w_small = ctx.verify_batch(*small, schnorr=True)
    w_large = ctx.verify_batch(*large)
    try:
        got, h = _dev_verify_pk(ks, *small, True)
        assert (got == w_small).all() and h == _host_hits(small[0], keys)
        # interleaved: general device verify on s1, pk verify on s2, keyed verify (by index) on s3
        s1, s2, s3 = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
        pk, flat, off, sg = large
        d_pk, d_msg, d_off, d_sig = _to_dev(dev, pk, flat, off, sg)
        n = pk.shape[0]
        d_st1 = torch.full((n,), 99, dtype=torch.uint8, device=dev)
        d_st2 = torch.full((n,), 99, dtype=torch.uint8, device=dev)
        d_hits = torch.full((1,), -1, dtype=torch.int64, device=dev)
        reg_rows = _rows(keys)
        mask = np.isin(_rows(pk), reg_rows)
        order = np.argsort(reg_rows)
        kidx = order[np.searchsorted(reg_rows[order], _rows(pk)[mask])].astype(np.uint32)
        sel = np.nonzero(mask)[0]
        sub_off = np.concatenate([[0], np.cumsum(np.diff(off)[sel])]).astype(np.uint64)
        sub_msg = flat.reshape(-1, 64)[sel].reshape(-1).copy()
        d_kidx, d_smsg, d_soff, d_ssig = _to_dev(dev, kidx.view(np.int32), sub_msg, sub_off, sg[sel].copy())
        d_st3 = torch.full((sel.size,), 99, dtype=torch.uint8, device=dev)
        for s in (s1, s2, s3):
            s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s1):
            ctx.dev_verify(n, d_pk, d_msg, d_off, d_sig, d_st1)
        with torch.cuda.stream(s2):
            ks.dev_verify_pk(n, d_pk, d_msg, d_off, d_sig, d_st2, hits=d_hits)
        with torch.cuda.stream(s3):
            ks.dev_verify(sel.size, d_kidx, d_smsg, d_soff, d_ssig, d_st3)
        torch.cuda.synchronize()
        assert (d_st1.cpu().numpy() == w_large).all()
        assert (d_st2.cpu().numpy() == w_large).all()
        assert int(d_hits.cpu()[0]) == int(mask.sum())
        assert (d_st3.cpu().numpy() == w_large[sel]).all()
        ctx.wipe()
        got, h = ks.verify_pk_batch(*small, schnorr=True, return_hits=True)
        assert (got == w_small).all() and h == _host_hits(small[0], keys)
        ctx.wipe()
        got, h = _dev_verify_pk(ks, *large, False)
        assert (got == w_large).all() and h == int(mask.sum())
    finally:
        ks.close()
    # the context still verifies after the set is gone
    assert (ctx.verify_batch(*small, schnorr=True) == w_small).all()


def test_pk_argument_errors(kb, ctx, mctx, registered, golden_records):
    """NULL pointers with n > 0, a NULL key set, decreasing message offsets: KB_ERR_ARG; n = 0: KB_OK, nothing written."""
    L = ctx.L
    a_reg, keys, ks, mks = registered[7]
    pk, flat, off, sg = _make_batch(ctx, a_reg, keys, 64, (1, 2), seed=11)
    st = np.full(64, 99, dtype=np.uint8)
    hits = np.full(1, 12345, dtype=np.uint64)
    p = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731
    args = [p(pk), p(flat), p(off), p(sg), p(st)]
    for k in range(5):
        if k == 1:
            continue   # msg may be NULL only when there are no message bytes
        a = list(args)
        a[k] = None
        assert L.kb_keyset_verify_pk_batch(ks.h, 64, *a, 0, p(hits)) == KB_ERR_ARG
        assert L.kb_mctx_keyset_verify_pk_batch(mks.h, 64, *a, 0, p(hits)) == KB_ERR_ARG
        assert L.kb_dev_keyset_verify_pk(ks.h, 64, *a, 0, None, None) == KB_ERR_ARG
    a = list(args)
    a[1] = None
    assert L.kb_keyset_verify_pk_batch(ks.h, 64, *a, 0, p(hits)) == KB_ERR_ARG
    assert L.kb_keyset_verify_pk_batch(None, 64, *args, 0, p(hits)) == KB_ERR_ARG
    assert L.kb_dev_keyset_verify_pk(None, 64, *args, 0, None, None) == KB_ERR_ARG
    assert L.kb_mctx_keyset_verify_pk_batch(None, 64, *args, 0, p(hits)) == KB_ERR_ARG
    bad_off = off.copy()
    bad_off[30] = bad_off[31] + 1
    with pytest.raises(kb.KBError):
        ks.verify_pk_batch(pk, flat, bad_off, sg)
    with pytest.raises(kb.KBError):
        mks.verify_pk_batch(pk, flat, bad_off, sg)
    assert (st == 99).all() and hits[0] == 12345
    # n = 0: nothing read, nothing written
    for fn, h in ((L.kb_keyset_verify_pk_batch, ks.h), (L.kb_mctx_keyset_verify_pk_batch, mks.h)):
        assert fn(h, 0, None, None, None, None, None, 1, p(hits)) == KB_OK
    assert L.kb_dev_keyset_verify_pk(ks.h, 0, None, None, None, None, None, 0, None, None) == KB_OK
    assert hits[0] == 12345
    # the set still works, and messages without bytes need no msg pointer
    e_off = np.zeros(3, dtype=np.uint64)
    want = ctx.verify_batch(pk[:2], np.zeros(0, dtype=np.uint8), e_off, sg[:2])
    assert (ks.verify_pk_batch(pk[:2], np.zeros(0, dtype=np.uint8), e_off, sg[:2]) == want).all()
    got, _ = _dev_verify_pk(ks, pk[:2], np.zeros(0, dtype=np.uint8), e_off, sg[:2], False)
    assert (got == want).all()


def test_pk_from_plain_c(kb, ctx, registered, tmp_path):
    """tests/c/keyset_pk_check.c: the three entry points from plain C (gcc, -lkyber_b200) on a fixture whose expected
    statuses and hit count come from the general verifier."""
    import subprocess

    a_reg, keys, _, _ = registered[7]
    pk, flat, off, sg = _make_batch(ctx, a_reg, keys, 3000, (1, 2), seed=21)
    want = [ctx.verify_batch(pk, flat, off, sg, schnorr=s) for s in (False, True)]
    fx = tmp_path / "fixture.bin"
    with open(fx, "wb") as f:
        f.write(np.array([pk.shape[0], flat.size, keys.shape[0], _host_hits(pk, keys)], dtype=np.uint64).tobytes())
        for a in (keys, pk, sg, off, flat, want[0].astype(np.uint8), want[1].astype(np.uint8)):
            f.write(np.ascontiguousarray(a).tobytes())
    exe = tmp_path / "keyset_pk_check"
    libdir = os.path.dirname(kb.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "keyset_pk_check.c"),
                           "-L", libdir, "-lkyber_b200", "-Wl,-rpath," + libdir, "-o", str(exe)])
    r = subprocess.run([str(exe), str(fx)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "mismatches=0" in r.stdout
