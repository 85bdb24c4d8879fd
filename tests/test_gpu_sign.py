"""Signing on the B200: kb_schnorr_sign_batch against the big-integer oracle and against the four-call composition it
replaces, signer sets (Schnorr and EdDSA) against the general signers, the device-buffer and multi-device forms, the
argument checks, and that every signature verifies under the library's verifiers."""
import ctypes
import importlib
import os
import subprocess

import numpy as np
import pytest

from helpers import ROOT, xof_bytes
from oracle import ed25519_bigint as O

pytestmark = pytest.mark.gpu

L = O.L
ERR_ARG = -1


@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


@pytest.fixture(scope="module")
def ctx(kb):
    c = kb.Context(0)
    yield c
    c.close()


def _sc(v):
    return int(v).to_bytes(32, "little")


def _arr(byte_list, width=32):
    return np.frombuffer(b"".join(byte_list), dtype=np.uint8).reshape(-1, width).copy()


def _rand(seed, n, width=32):
    return np.frombuffer(xof_bytes(seed, width * n), dtype=np.uint8).reshape(n, width).copy()


def _pack(msgs):
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs])
    flat = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy() if off[-1] else np.zeros(0, dtype=np.uint8)
    return flat, off


def _msgs_of(n, seed, lens):
    blob = xof_bytes(seed, int(sum(lens)))
    out, p = [], 0
    for ln in lens:
        out.append(blob[p:p + ln])
        p += ln
    return out


def _schnorr_keys(golden_records, k):
    """k secret scalars: reduced ones, clamped unreduced keys (bit 254 set, as curve.rs:74-87 derives them) and the edges
    0, 1, L-1, L."""
    edge = [_sc(0), _sc(1), _sc(L - 1), _sc(L)]
    clamped = [O.clamp_key(r[0])[0] for r in golden_records[:max(0, k // 3)]]
    red = [O.scalar_set_bytes(xof_bytes(f"kyber-b200/test/sign/x{i}", 64)) for i in range(k)]
    return (edge + clamped + red)[:k]


def _verify_all(ctx, sig, pk, flat, off, good):
    """status 0 under both general verifiers and under a key set built from the distinct public keys, for the items in good"""
    for schnorr in (False, True):
        st = ctx.verify_batch(pk, flat, off, sig, schnorr=schnorr)
        assert not st[good].any(), np.nonzero(st[good])[0][:10]
    keys, key_idx = np.unique(pk, axis=0, return_inverse=True)
    ks = ctx.keyset(keys)
    try:
        for schnorr in (False, True):
            st = ks.verify_batch(key_idx.astype(np.uint32).ravel(), flat, off, sig, schnorr=schnorr)
            assert not st[good].any(), np.nonzero(st[good])[0][:10]
    finally:
        ks.close()


# SHA-512 padding edges of 64 + len bytes (R || A || M): 47, 48 (one block), 64, 175, 176, 192, plus 0, 1, 8 KiB and one
# message of the size of a bincode deal at t = 683 (about 110 KiB)
LENS = [47, 48, 64, 175, 176, 192, 0, 1, 8192]
DEAL_LEN = 110 * 1024 + 37


def test_schnorr_sign_against_oracle(ctx, golden_records):
    secrets = _schnorr_keys(golden_records, 13)
    nonces = [_sc(0), _sc(1), _sc(L - 1)] + [O.scalar_set_bytes(xof_bytes(f"kyber-b200/test/sign/k{i}", 64)) for i in range(4)]
    n = 320
    xs = [secrets[i % len(secrets)] for i in range(n)]
    ks = [nonces[(i // len(secrets)) % len(nonces)] for i in range(n)]
    lens = [LENS[i % len(LENS)] for i in range(n)]
    lens[123] = DEAL_LEN
    msgs = _msgs_of(n, "kyber-b200/test/sign/oracle-msgs", lens)
    flat, off = _pack(msgs)
    sig, pk = ctx.schnorr_sign_batch(_arr(xs), _arr(ks), flat, off)
    for i in range(n):
        assert sig[i].tobytes() == O.schnorr_sign(xs[i], msgs[i], ks[i]), i
        assert pk[i].tobytes() == O.point_encode(O.point_mul(xs[i])), i
    # R or A is the identity when k or x is a multiple of L: the verifiers reject those as the oracle does
    degenerate = np.array([int.from_bytes(x, "little") % L == 0 or int.from_bytes(k, "little") % L == 0 for x, k in zip(xs, ks)])
    assert degenerate.any() and not degenerate.all()
    _verify_all(ctx, sig, pk, flat, off, ~degenerate)
    st = ctx.verify_batch(pk, flat, off, sig, schnorr=True)
    for i in np.nonzero(degenerate)[0][:8]:
        assert st[i] == O.schnorr_verify(pk[i].tobytes(), msgs[i], sig[i].tobytes()) != 0


def test_schnorr_sign_against_composition_at_size(ctx, golden_records):
    """2^20 + 37 items, nonces with byte 31 > 127 among them: byte for byte the four calls it replaces (constant-time x*B and
    k*B, challenge, sc_muladd); every item with an in-domain nonce verifies."""
    n = (1 << 20) + 37
    nkeys = 1024
    keys = _arr(_schnorr_keys(golden_records, nkeys - 4) + [_sc(L + 5), _sc(3 * L), _sc(2**255 - 19), _sc(2**256 - 1)])
    key_idx = (np.arange(n, dtype=np.uint64) * 2654435761 % nkeys).astype(np.uint32)
    x = keys[key_idx]
    k = _rand("kyber-b200/test/sign/comp-nonces", n)
    k[:, 31] &= 0x7F
    k[::97, 31] |= 0x80   # out of the domain of the fixed-base multiplication
    lens = (np.arange(n) * 7 % 160).tolist()
    flat = np.frombuffer(xof_bytes("kyber-b200/test/sign/comp-msgs", int(sum(lens))), dtype=np.uint8).copy()
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum(lens)
    sig, pk = ctx.schnorr_sign_batch(x, k, flat, off)
    A = ctx.point_mul_base_batch(x)
    R = ctx.point_mul_base_batch(k)
    h = ctx.challenge_batch(R, A, flat, off)
    s = ctx.sc_muladd_batch(x, h, k)
    assert (pk == A).all()
    assert (sig[:, :32] == R).all() and (sig[:, 32:] == s).all(), np.nonzero((sig != np.concatenate([R, s], axis=1)).any(axis=1))[0][:10]
    zero = np.array([int.from_bytes(kk.tobytes(), "little") % L == 0 for kk in keys])   # 0, L, 3L: A is the identity
    good = (k[:, 31] <= 127) & (x[:, 31] <= 127) & ~zero[key_idx]
    _verify_all(ctx, sig, pk, flat, off, good)


@pytest.mark.parametrize("nkeys", [1, 7, 1024])
def test_schnorr_signer_set(ctx, golden_records, nkeys):
    keys = _arr(_schnorr_keys(golden_records, nkeys)) if nkeys != 7 else _arr(_schnorr_keys(golden_records, 6) + [_sc(2**256 - 1)])
    n = 20011 if nkeys == 1024 else 3001
    rng = np.random.default_rng(nkeys)
    key_idx = rng.integers(0, nkeys, size=n, dtype=np.uint32)
    nonces = _rand(f"kyber-b200/test/sign/set-nonces/{nkeys}", n)
    nonces[::5, 31] &= 0x7F
    msgs = _msgs_of(n, f"kyber-b200/test/sign/set-msgs/{nkeys}", (np.arange(n) * 13 % 300).tolist())
    flat, off = _pack(msgs)
    want, want_pk = ctx.schnorr_sign_batch(keys[key_idx], nonces, flat, off)
    ss = ctx.signerset(keys)
    try:
        assert (ss.pk == ctx.point_mul_base_batch(keys)).all()
        sig = ss.sign_batch(key_idx, flat, off, nonces)
        assert (sig == want).all(), np.nonzero((sig != want).any(axis=1))[0][:10]
        d_sig, d_st = _dev_sign(ss, key_idx, nonces, flat, off)
        assert (d_sig == want).all() and not d_st.any()
    finally:
        ss.close()


def test_eddsa_signer_set_golden(kb, ctx, golden_records):
    """The 1024 seeds of the reference's sign.input as one set: signing the 1024 messages in a shuffled order reproduces
    every golden signature; repeated indices equal kb_eddsa_sign_batch on seeds[key_idx]."""
    seeds = _arr([r[0] for r in golden_records])
    gold_pk = _arr([r[1] for r in golden_records])
    gold_sig = _arr([r[2] for r in golden_records], 64)
    msgs = [r[3] for r in golden_records]
    ss = ctx.signerset(seeds, kb.SIGNER_EDDSA)
    try:
        assert (ss.pk == gold_pk).all()
        perm = np.random.default_rng(5).permutation(1024).astype(np.uint32)
        flat, off = _pack([msgs[i] for i in perm])
        sig = ss.sign_batch(perm, flat, off)
        assert (sig == gold_sig[perm]).all()
        d_sig, d_st = _dev_sign(ss, perm, None, flat, off)
        assert (d_sig == gold_sig[perm]).all() and not d_st.any()
        n = 5000
        key_idx = np.random.default_rng(6).integers(0, 8, size=n, dtype=np.uint32) * 131
        mm = _msgs_of(n, "kyber-b200/test/sign/eddsa-rep", (np.arange(n) * 11 % 400).tolist())
        flat, off = _pack(mm)
        want, _ = ctx.eddsa_sign_batch(seeds[key_idx], flat, off)
        assert (ss.sign_batch(key_idx, flat, off) == want).all()
        assert not ctx.verify_batch(ss.pk[key_idx], flat, off, want).any()
    finally:
        ss.close()


def _to_dev(*arrays):
    import torch

    dev = torch.device("cuda", 0)
    return [torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a.view(np.int64) if a.dtype == np.uint64 else a).to(dev) if a is not None else None for a in arrays]


def _dev_sign(ss, key_idx, nonces, flat, off):
    import torch

    n = key_idx.shape[0]
    d_idx, d_k, d_m, d_off = _to_dev(key_idx, nonces, flat if flat.size else np.zeros(1, np.uint8), off)
    d_sig = torch.full((n, 64), 0xAA, dtype=torch.uint8, device=d_off.device)
    d_st = torch.full((n,), 99, dtype=torch.uint8, device=d_off.device)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ss.dev_sign(n, d_idx, d_k, d_m, d_off, d_sig, d_st)
    s.synchronize()
    return d_sig.cpu().numpy(), d_st.cpu().numpy()


def test_device_buffers(kb, ctx, golden_records):
    """kb_dev_schnorr_sign equals the host call; an index outside a set gives status 0xFF and 64 zero bytes on the device
    form, the other items are unchanged, for both kinds."""
    import torch

    n = 4099
    keys = _arr(_schnorr_keys(golden_records, 9))
    key_idx = np.random.default_rng(2).integers(0, 9, size=n, dtype=np.uint32)
    x, k = keys[key_idx], random_in_domain("kyber-b200/test/sign/dev-k", n)
    msgs = _msgs_of(n, "kyber-b200/test/sign/dev-msgs", (np.arange(n) * 5 % 250).tolist())
    flat, off = _pack(msgs)
    want, want_pk = ctx.schnorr_sign_batch(x, k, flat, off)
    d_x, d_k, d_m, d_off = _to_dev(x, k, flat, off)
    d_sig = torch.empty((n, 64), dtype=torch.uint8, device=d_x.device)
    d_pk = torch.empty((n, 32), dtype=torch.uint8, device=d_x.device)
    ctx.dev_schnorr_sign(n, d_x, d_k, d_m, d_off, d_sig, d_pk)
    torch.cuda.synchronize()
    assert (d_sig.cpu().numpy() == want).all() and (d_pk.cpu().numpy() == want_pk).all()
    ctx.dev_schnorr_sign(n, d_x, d_k, d_m, d_off, d_sig, None)
    torch.cuda.synchronize()
    assert (d_sig.cpu().numpy() == want).all()
    bad = key_idx.copy()
    bad[[7, 4000]] = [9, 0xFFFFFFFF]
    keep = np.ones(n, dtype=bool)
    keep[[7, 4000]] = False
    seeds = _arr([r[0] for r in golden_records[:9]])
    for kind, kk, ref in ((kb.SIGNER_SCHNORR, k, want), (kb.SIGNER_EDDSA, None, ctx.eddsa_sign_batch(seeds[key_idx], flat, off)[0])):
        ss = ctx.signerset(keys if kind == kb.SIGNER_SCHNORR else seeds, kind)
        try:
            sig, st = _dev_sign(ss, bad, kk, flat, off)
            assert (st[~keep] == 0xFF).all() and not sig[~keep].any()
            assert not st[keep].any() and (sig[keep] == ref[keep]).all()
        finally:
            ss.close()


def random_in_domain(seed, n):
    k = _rand(seed, n)
    k[:, 31] &= 0x7F
    return k


def _call(fn, *args):
    conv = [ctypes.c_void_p(a.ctypes.data) if isinstance(a, np.ndarray) else a for a in args]
    return fn(*conv)


def test_argument_errors(kb, ctx, golden_records):
    """KB_ERR_ARG with the outputs untouched for an index >= nkeys, a Schnorr set without nonces, an EdDSA set with nonces
    and a decreasing msg_off; n = 0 is KB_OK; two sets on one context, created and destroyed in either order."""
    Lb = ctx.L
    n = 64
    keys = _arr(_schnorr_keys(golden_records, 5))
    seeds = _arr([r[0] for r in golden_records[:5]])
    key_idx = (np.arange(n) % 5).astype(np.uint32)
    k = random_in_domain("kyber-b200/test/sign/args-k", n)
    flat, off = _pack(_msgs_of(n, "kyber-b200/test/sign/args-msgs", [40] * n))
    want_s, _ = ctx.schnorr_sign_batch(keys[key_idx], k, flat, off)
    want_e, _ = ctx.eddsa_sign_batch(seeds[key_idx], flat, off)
    a = ctx.signerset(keys)
    b = ctx.signerset(seeds, kb.SIGNER_EDDSA)
    sig = np.full((n, 64), 0xAA, dtype=np.uint8)
    pk = np.full((n, 32), 0xAA, dtype=np.uint8)
    try:
        badidx = key_idx.copy()
        badidx[9] = 5
        decreasing = off.copy()
        decreasing[10] = decreasing[11] + 1
        assert _call(Lb.kb_signerset_sign_batch, a.h, n, badidx, k, flat, off, sig) == ERR_ARG
        assert _call(Lb.kb_signerset_sign_batch, b.h, n, badidx, None, flat, off, sig) == ERR_ARG
        assert _call(Lb.kb_signerset_sign_batch, a.h, n, key_idx, None, flat, off, sig) == ERR_ARG
        assert _call(Lb.kb_signerset_sign_batch, b.h, n, key_idx, k, flat, off, sig) == ERR_ARG
        assert _call(Lb.kb_signerset_sign_batch, a.h, n, key_idx, k, flat, decreasing, sig) == ERR_ARG
        assert _call(Lb.kb_schnorr_sign_batch, ctx.h, n, keys[key_idx], k, flat, decreasing, sig, pk) == ERR_ARG
        assert _call(Lb.kb_schnorr_sign_batch, ctx.h, n, keys[key_idx], None, flat, off, sig, pk) == ERR_ARG
        assert (sig == 0xAA).all() and (pk == 0xAA).all()
        assert Lb.kb_dev_signerset_sign(a.h, 0, None, None, None, None, None, None, None) == ERR_ARG   # Schnorr set without nonces
        assert Lb.kb_dev_signerset_sign(b.h, 0, None, None, None, None, None, None, None) == 0
        assert _call(Lb.kb_signerset_sign_batch, a.h, 0, None, k, None, None, None) == 0
        assert _call(Lb.kb_schnorr_sign_batch, ctx.h, 0, None, None, None, None, None, None) == 0
        assert _call(Lb.kb_signerset_create, ctx.h, 5, keys, 2, None, ctypes.byref(ctypes.c_void_p())) == ERR_ARG
        assert _call(Lb.kb_signerset_create, ctx.h, 0, keys, 0, None, ctypes.byref(ctypes.c_void_p())) == ERR_ARG
        assert (a.sign_batch(key_idx, flat, off, k) == want_s).all() and (b.sign_batch(key_idx, flat, off) == want_e).all()
        a.close()   # created first, destroyed first
        assert (b.sign_batch(key_idx, flat, off) == want_e).all()
        c = ctx.signerset(keys)
        b.close()   # created first, destroyed before the later one
        assert (c.sign_batch(key_idx, flat, off, k) == want_s).all()
        c.close()
    finally:
        a.close()
        b.close()
    d = ctx.signerset(keys)
    try:
        with pytest.raises(kb.KBError):
            d.sign_batch(key_idx, flat, off)
    finally:
        d.close()


_LAYOUT = r"""
#define KB_HOST_EMU 1
#include <stddef.h>
#include "ctx.cuh"
int main() { printf("%zu %zu\n", offsetof(kb_ctx, slot), offsetof(kb_ctx, slot_bytes)); return 0; }
"""


def _scratch_slot(ctx, tmp_path, s):
    """Bytes of scratch slot s of the context: the slot's device pointer and size read from the kb_ctx struct (offsets from a
    host build of csrc/ctx.cuh), copied with the driver API."""
    src = tmp_path / "layout.cpp"
    src.write_text(_LAYOUT)
    exe = tmp_path / "layout"
    subprocess.check_call(["g++", "-std=c++17", "-I/usr/local/cuda/include", "-I", os.path.join(ROOT, "kyber-rs_b200", "csrc"), "-o", str(exe), str(src)])
    off_slot, off_bytes = (int(v) for v in subprocess.check_output([str(exe)]).split())
    base = ctx.h.value
    ptr = ctypes.c_uint64.from_address(base + off_slot + 8 * s).value
    size = ctypes.c_size_t.from_address(base + off_bytes + 8 * s).value
    assert ptr and size
    cu = ctypes.CDLL("libcuda.so.1")
    buf = ctypes.create_string_buffer(size)
    assert cu.cuMemcpyDtoH_v2(buf, ctypes.c_uint64(ptr), ctypes.c_size_t(size)) == 0
    return buf.raw


def test_secrets_leave_no_trace_in_scratch(kb, golden_records, tmp_path):
    """The host forms zero the scratch slots that held secrets and nonces (0 and 6 for kb_schnorr_sign_batch, 6 for a Schnorr
    set, 9 for the nonces an EdDSA set derives) before they return."""
    c = kb.Context(0)
    try:
        n = 3000
        keys = _arr(_schnorr_keys(golden_records, 7))
        key_idx = (np.arange(n) % 7).astype(np.uint32)
        k = random_in_domain("kyber-b200/test/sign/scratch-k", n)
        flat, off = _pack(_msgs_of(n, "kyber-b200/test/sign/scratch-msgs", [64] * n))
        c.schnorr_sign_batch(keys[key_idx], k, flat, off)
        assert _scratch_slot(c, tmp_path, 0)[:32 * n] == bytes(32 * n)
        assert _scratch_slot(c, tmp_path, 6)[:32 * n] == bytes(32 * n)
        ss = c.signerset(keys)
        es = c.signerset(_arr([r[0] for r in golden_records[:7]]), kb.SIGNER_EDDSA)
        try:
            ss.sign_batch(key_idx, flat, off, k)
            assert _scratch_slot(c, tmp_path, 6)[:32 * n] == bytes(32 * n)
            es.sign_batch(key_idx, flat, off)
            assert _scratch_slot(c, tmp_path, 9)[:32 * n] == bytes(32 * n)
        finally:
            es.close()
            ss.close()
    finally:
        c.close()


@pytest.mark.parametrize("which", ["one", "all"])
def test_multi_device(kb, ctx, golden_records, which):
    """kb_mctx_schnorr_sign_batch and the kb_mctx signer sets give the bytes of one device, on as many GPUs as are visible; a
    bad index or nonce / kind pairing is refused before any device starts."""
    import torch

    ngpu = torch.cuda.device_count()
    if which == "all" and ngpu < 2:
        pytest.skip("a single GPU is visible")
    devs = [0] if which == "one" else list(range(min(ngpu, 8)))
    n = 10007
    keys = _arr(_schnorr_keys(golden_records, 11))
    seeds = _arr([r[0] for r in golden_records[:11]])
    key_idx = np.random.default_rng(8).integers(0, 11, size=n, dtype=np.uint32)
    k = random_in_domain("kyber-b200/test/sign/multi-k", n)
    flat, off = _pack(_msgs_of(n, "kyber-b200/test/sign/multi-msgs", (np.arange(n) * 3 % 200).tolist()))
    want, want_pk = ctx.schnorr_sign_batch(keys[key_idx], k, flat, off)
    want_e, _ = ctx.eddsa_sign_batch(seeds[key_idx], flat, off)
    m = kb.MultiContext(devs)
    try:
        sig, pk = m.schnorr_sign_batch(keys[key_idx], k, flat, off)
        assert (sig == want).all() and (pk == want_pk).all()
        ms = m.signerset(keys)
        me = m.signerset(seeds, kb.SIGNER_EDDSA)
        try:
            assert (ms.pk == ctx.point_mul_base_batch(keys)).all()
            assert (ms.sign_batch(key_idx, flat, off, k) == want).all()
            assert (me.sign_batch(key_idx, flat, off) == want_e).all()
            bad = key_idx.copy()
            bad[-1] = 11
            with pytest.raises(kb.KBError):
                ms.sign_batch(bad, flat, off, k)
            with pytest.raises(kb.KBError):
                me.sign_batch(key_idx, flat, off, k)
        finally:
            me.close()
            ms.close()
    finally:
        m.close()


def test_host_schnorr_sign_is_one_call(kb, ctx):
    """host.schnorr_sign_batch launches exactly the three kernels of kb_schnorr_sign_batch."""
    priv = [O.scalar_set_bytes(xof_bytes(f"kyber-b200/test/sign/h{i}", 64)) for i in range(8)]
    nonce = [O.scalar_set_bytes(xof_bytes(f"kyber-b200/test/sign/hk{i}", 64)) for i in range(8)]
    msgs = [b"m" * i for i in range(8)]
    before = ctx.launches
    sigs, _ = kb.host.schnorr_sign_batch(priv, msgs, nonce, ctx=ctx)
    assert ctx.launches - before == 3
    for i in range(8):
        assert sigs[i].tobytes() == O.schnorr_sign(priv[i], msgs[i], nonce[i])


def test_sign_from_plain_c(kb, ctx, golden_records, tmp_path):
    """tests/c/sign_check.c: kb_schnorr_sign_batch and a Schnorr signer set from plain C (gcc, -lkyber_b200), on a fixture
    whose expected bytes come from the Python binding."""
    nkeys, n = 7, 2000
    keys = _arr(_schnorr_keys(golden_records, nkeys))
    key_idx = np.random.default_rng(12).integers(0, nkeys, size=n, dtype=np.uint32)
    k = random_in_domain("kyber-b200/test/sign/c-k", n)
    flat, off = _pack(_msgs_of(n, "kyber-b200/test/sign/c-msgs", (np.arange(n) * 17 % 230).tolist()))
    want, _ = ctx.schnorr_sign_batch(keys[key_idx], k, flat, off)
    want_pk = ctx.point_mul_base_batch(keys)
    fx = tmp_path / "fixture.bin"
    with open(fx, "wb") as f:
        f.write(np.array([n, nkeys], dtype=np.uint64).tobytes())
        for a in (keys, key_idx, k, off, flat, want, want_pk):
            f.write(np.ascontiguousarray(a).tobytes())
    exe = tmp_path / "sign_check"
    libdir = os.path.dirname(kb.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "sign_check.c"),
                           "-L", libdir, "-lkyber_b200", "-Wl,-rpath," + libdir, "-o", str(exe)])
    r = subprocess.run([str(exe), str(fx)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "mismatches=0" in r.stdout
