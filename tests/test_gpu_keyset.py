"""Key sets on the B200: kb_keyset_verify_batch / kb_dev_keyset_verify return, item for item, what the general verifiers
(and the C oracle) return for pk = keys[key_idx[i]]."""
import importlib

import numpy as np
import pytest

from helpers import make_mixed_order_sigs, make_sig_batch, pack_batch, xof_bytes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


@pytest.fixture(scope="module")
def ctx(kb):
    c = kb.Context(0)
    yield c
    c.close()


def _index_keys(pk):
    """(keys, key_idx) with keys[key_idx] == pk: every distinct key once, in order of first appearance."""
    keys, first, inv = np.unique(pk, axis=0, return_index=True, return_inverse=True)
    order = np.argsort(first)
    rank = np.empty_like(order)
    rank[order] = np.arange(order.size)
    return keys[order], rank[inv.reshape(-1)].astype(np.uint32)


def _to_dev(dev, *arrays):
    import torch

    out = []
    for a in arrays:
        if a.dtype == np.uint64:
            a = a.view(np.int64)
        elif a.dtype == np.uint32:
            a = a.view(np.int32)
        out.append(torch.from_numpy(a if a.size else np.zeros(1, dtype=a.dtype)).to(dev))
    return out


def _dev_verify(ks, key_idx, flat, off, sg, schnorr, stream=None):
    import torch

    dev = torch.device("cuda", 0)
    n = key_idx.shape[0]
    d_idx, d_msg, d_off, d_sig = _to_dev(dev, key_idx, flat, off, sg)
    d_st = torch.full((max(n, 1),), 99, dtype=torch.uint8, device=dev)
    s = stream if stream is not None else torch.cuda.current_stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ks.dev_verify(n, d_idx, d_msg, d_off, d_sig, d_st, schnorr=schnorr)
    s.synchronize()
    return d_st.cpu().numpy()[:n]


@pytest.mark.parametrize("schnorr", [False, True])
def test_keyset_matches_general_verifier_and_oracle(ctx, coracle, golden_records, schnorr):
    """Golden records with every mutation class (mutated keys become keys of the set) and signatures under keys with a
    small-order component, accepted and near misses."""
    good, bad = make_mixed_order_sigs(48, seed=13)
    pks, msgs, sigs = make_sig_batch(golden_records, 3000, bad_every=2)
    pks += [x[0] for x in good + bad]
    msgs += [x[1] for x in good + bad]
    sigs += [x[2] for x in good + bad]
    pk, flat, off, sg = pack_batch(pks, msgs, sigs)
    keys, key_idx = _index_keys(pk)
    assert (keys[key_idx] == pk).all()
    want = coracle.verify_batch(pk, flat, off, sg, nthreads=8, schnorr=schnorr)
    assert set(np.unique(want)) == {0, 2, 3, 4, 5, 6, 7, 8}
    assert (ctx.verify_batch(pk, flat, off, sg, schnorr=schnorr) == want).all()
    ks = ctx.keyset(keys)
    try:
        got = ks.verify_batch(key_idx, flat, off, sg, schnorr=schnorr)
        assert (got == want).all(), np.nonzero(got != want)[0][:10]
        got = _dev_verify(ks, key_idx, flat, off, sg, schnorr)
        assert (got == want).all(), np.nonzero(got != want)[0][:10]
    finally:
        ks.close()


def _signed_batch(ctx, nkeys, n, seed):
    """n fresh signatures (64-byte messages) under nkeys keys with random key_idx; 1/8 damaged in s, R or the message."""
    rng = np.random.default_rng(seed)
    kseeds = np.frombuffer(xof_bytes(f"kyber-b200/test/keyset/{seed}/{nkeys}", 32 * nkeys), dtype=np.uint8).reshape(nkeys, 32)
    key_idx = rng.integers(0, nkeys, size=n, dtype=np.uint32)
    flat = np.frombuffer(xof_bytes(f"kyber-b200/test/keyset/msg/{seed}", 64 * n), dtype=np.uint8).copy()
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(64)
    sigs, pks = ctx.eddsa_sign_batch(kseeds[key_idx], flat, off)
    sigs, pks = sigs.copy(), pks.copy()
    for i in range(0, n, 8):
        kind = (i // 8) % 3
        if kind == 0:
            sigs[i, 32 + rng.integers(0, 31)] ^= 1 << rng.integers(0, 8)
        elif kind == 1:
            sigs[i, rng.integers(0, 32)] ^= 1 << rng.integers(0, 8)
        else:
            flat[64 * i + rng.integers(0, 64)] ^= 1
    keys = np.empty((nkeys, 32), dtype=np.uint8)
    keys[key_idx] = pks
    return keys, key_idx, pks, flat, off, sigs


@pytest.mark.parametrize("nkeys", [1, 7, 1024])
def test_keyset_large_batch(ctx, coracle, nkeys):
    """2^18 signatures under K keys through the host path and the device path (on a non-default stream)."""
    import torch

    n = 1 << 18
    keys, key_idx, pks, flat, off, sigs = _signed_batch(ctx, nkeys, n, seed=nkeys)
    used = np.unique(key_idx)
    if nkeys > 1:
        assert used.size == nkeys
    ks = ctx.keyset(keys)
    side = torch.cuda.Stream()
    try:
        for schnorr in (False, True):
            want = ctx.verify_batch(pks, flat, off, sigs, schnorr=schnorr)
            assert (want.reshape(-1, 8)[:, 1:] == 0).all() and want.reshape(-1, 8)[:, 0].all()
            m = 2048
            assert (want[:m] == coracle.verify_batch(pks[:m], flat[:64 * m], off[:m + 1], sigs[:m], nthreads=8, schnorr=schnorr)).all()
            got = ks.verify_batch(key_idx, flat, off, sigs, schnorr=schnorr)
            assert (got == want).all(), np.nonzero(got != want)[0][:10]
            got = _dev_verify(ks, key_idx, flat, off, sigs, schnorr, stream=side)
            assert (got == want).all(), np.nonzero(got != want)[0][:10]
    finally:
        ks.close()


def test_keyset_message_lengths(ctx, coracle, golden_records):
    """Empty messages and messages longer than one SHA-512 block (signed on the device)."""
    rng = np.random.default_rng(3)
    lens = [0, 0, 1, 63, 64, 111, 112, 127, 128, 129, 200, 1000, 4096] * 8
    n = len(lens)
    nkeys = 5
    kseeds = np.frombuffer(xof_bytes("kyber-b200/test/keyset/lens", 32 * nkeys), dtype=np.uint8).reshape(nkeys, 32)
    key_idx = rng.integers(0, nkeys, size=n, dtype=np.uint32)
    msgs = [bytes(rng.integers(0, 256, size=m, dtype=np.uint8)) for m in lens]
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum(lens)
    flat = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy()
    sigs, pks = ctx.eddsa_sign_batch(kseeds[key_idx], flat, off)
    sigs = sigs.copy()
    sigs[1::3, 40] ^= 2
    keys = np.empty((nkeys, 32), dtype=np.uint8)
    keys[key_idx] = pks
    ks = ctx.keyset(keys)
    try:
        for schnorr in (False, True):
            want = coracle.verify_batch(pks, flat, off, sigs, nthreads=4, schnorr=schnorr)
            assert (want[0::3] == 0).all() and (want[1::3] != 0).all()
            assert (ks.verify_batch(key_idx, flat, off, sigs, schnorr=schnorr) == want).all()
            assert (_dev_verify(ks, key_idx, flat, off, sigs, schnorr) == want).all()
        # only empty messages: no message bytes at all
        e_off = np.zeros(3, dtype=np.uint64)
        e_idx = key_idx[:2]
        assert lens[0] == lens[1] == 0
        want = coracle.verify_batch(pks[:2], flat[:0], e_off, sigs[:2], nthreads=1)
        assert (ks.verify_batch(e_idx, np.zeros(0, dtype=np.uint8), e_off, sigs[:2]) == want).all()
        assert (_dev_verify(ks, e_idx, np.zeros(0, dtype=np.uint8), e_off, sigs[:2], False) == want).all()
    finally:
        ks.close()


def test_keyset_argument_errors(kb, ctx, golden_records):
    """key_idx >= nkeys: KBError on the host path, status 0xFF for exactly those items on the device path; n = 0; nkeys = 0."""
    pks, msgs, sigs = make_sig_batch(golden_records[:64], 200, bad_every=5)
    pk, flat, off, sg = pack_batch(pks, msgs, sigs)
    keys, key_idx = _index_keys(pk)
    want = ctx.verify_batch(pk, flat, off, sg)
    ks = ctx.keyset(keys)
    try:
        bad = key_idx.copy()
        bad[17] = keys.shape[0]
        with pytest.raises(kb.KBError):
            ks.verify_batch(bad, flat, off, sg)
        bad[101] = 0xFFFFFFFF
        got = _dev_verify(ks, bad, flat, off, sg, False)
        assert got[17] == 0xFF and got[101] == 0xFF
        keep = np.ones(200, dtype=bool)
        keep[[17, 101]] = False
        assert (got[keep] == want[keep]).all()
        assert (ks.verify_batch(key_idx, flat, off, sg) == want).all()   # still usable
        # n = 0
        e = np.zeros(0, dtype=np.uint32)
        assert ks.verify_batch(e, np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.uint64), np.zeros((0, 64), dtype=np.uint8)).shape == (0,)
        assert _dev_verify(ks, e, np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.uint64), np.zeros((0, 64), dtype=np.uint8), True).shape == (0,)
    finally:
        ks.close()
    with pytest.raises(kb.KBError):
        ctx.keyset(np.zeros((0, 32), dtype=np.uint8))


def test_two_keysets_scratch_growth_and_wipe(ctx, coracle, golden_records):
    """Two key sets on one context, interleaved with a larger kb_dev_eddsa_verify that grows the scratch; destroying one
    leaves the other correct; a key set still verifies after kb_ctx_wipe (its combs are not scratch)."""
    import torch

    dev = torch.device("cuda", 0)
    pa, ma, sa = make_sig_batch(golden_records[:300], 600, bad_every=3)
    pb, mb, sb = make_sig_batch(golden_records[500:900], 700, bad_every=4)
    A = pack_batch(pa, ma, sa)
    B = pack_batch(pb, mb, sb)
    wa = coracle.verify_batch(*A, nthreads=8)
    wb = coracle.verify_batch(*B, nthreads=8, schnorr=True)
    ka, ia = _index_keys(A[0])
    kb_, ib = _index_keys(B[0])
    ks_a, ks_b = ctx.keyset(ka), ctx.keyset(kb_)
    try:
        assert (_dev_verify(ks_a, ia, *A[1:], False) == wa).all()
        # a general device verify four times larger than anything before: the scratch slots grow
        pk, flat, off, sg = pack_batch(*make_sig_batch(golden_records, 50000, bad_every=6))
        d_pk, d_msg, d_off, d_sig = _to_dev(dev, pk, flat, off, sg)
        d_st = torch.full((pk.shape[0],), 99, dtype=torch.uint8, device=dev)
        ctx.dev_verify(pk.shape[0], d_pk, d_msg, d_off, d_sig, d_st)
        assert (_dev_verify(ks_b, ib, *B[1:], True) == wb).all()
        torch.cuda.synchronize()
        assert (d_st.cpu().numpy()[:3000] == coracle.verify_batch(pk[:3000], flat, off[:3001], sg[:3000], nthreads=8)).all()
        assert (ks_a.verify_batch(ia, *A[1:]) == wa).all()
        ks_a.close()
        assert (ks_b.verify_batch(ib, *B[1:], schnorr=True) == wb).all()
        assert (_dev_verify(ks_b, ib, *B[1:], True) == wb).all()
        ctx.wipe()
        assert (ks_b.verify_batch(ib, *B[1:], schnorr=True) == wb).all()
        assert (_dev_verify(ks_b, ib, *B[1:], True) == wb).all()
    finally:
        ks_a.close()
        ks_b.close()


def test_keyset_from_plain_c(kb, coracle, golden_records, tmp_path):
    """tests/c/keyset_check.c: create / verify (EdDSA and Schnorr) / destroy from plain C (gcc, -lkyber_b200), on a
    fixture whose expected statuses come from the oracle."""
    import os
    import subprocess

    from helpers import ROOT

    pks, msgs, sigs = make_sig_batch(golden_records, 1500, bad_every=3)
    pk, flat, off, sg = pack_batch(pks, msgs, sigs)
    keys, key_idx = _index_keys(pk)
    want = [coracle.verify_batch(pk, flat, off, sg, nthreads=8, schnorr=s) for s in (False, True)]
    fx = tmp_path / "fixture.bin"
    with open(fx, "wb") as f:
        f.write(np.array([pk.shape[0], flat.size, keys.shape[0]], dtype=np.uint64).tobytes())
        for a in (keys, key_idx, sg, off, flat, want[0].astype(np.uint8), want[1].astype(np.uint8)):
            f.write(np.ascontiguousarray(a).tobytes())
    exe = tmp_path / "keyset_check"
    libdir = os.path.dirname(kb.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "keyset_check.c"),
                           "-L", libdir, "-lkyber_b200", "-Wl,-rpath," + libdir, "-o", str(exe)])
    r = subprocess.run([str(exe), str(fx)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "mismatches=0" in r.stdout
