"""Keyed scalar multiplication on the B200: kb_keyset_mul_batch / kb_dev_keyset_mul / kb_mctx_keyset_mul_batch return, byte for
byte and status for status, what kb_point_mul_batch returns for points = keys[key_idx] (and what the C oracle returns)."""
import ctypes
import importlib
import os
import subprocess

import numpy as np
import pytest

from helpers import NONCANONICAL, ROOT, WEAK_KEYS, _off_curve, xof_bytes
from test_emu_keyset_mul import _torsion_key, noncanonical_keys, scalar_classes

pytestmark = pytest.mark.gpu

FLAGS = [0, 1]   # 0 and KB_FLAG_VARTIME


@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


@pytest.fixture(scope="module")
def ctx(kb):
    c = kb.Context(0)
    yield c
    c.close()


def _arr(byte_list):
    return np.frombuffer(b"".join(byte_list), dtype=np.uint8).reshape(-1, 32).copy()


def _key_classes(golden_records, coracle):
    """Golden keys, keys with a small-order component, the weak keys, non-canonical encodings that decode, encodings in the
    is_canonical quirk range, and encodings that do not decode."""
    keys = [r[1] for r in golden_records[:12]]
    keys += [_torsion_key(golden_records[20 + k][1], k) for k in range(1, 8)]
    keys += WEAK_KEYS + noncanonical_keys(coracle)
    keys += [bytes([0x20]) + b"\xff" * 30 + b"\x7f", bytes([0x20]) + b"\xff" * 30 + b"\xff", NONCANONICAL, _off_curve(7), _off_curve(8), _off_curve(9)]
    return _arr(keys)


def _to_dev(*arrays):
    import torch

    dev = torch.device("cuda", 0)
    return [torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a).to(dev) for a in arrays]


def _dev_mul(ks, key_idx, scalars, flags, stream=None):
    import torch

    n = key_idx.shape[0]
    d_idx, d_s = _to_dev(key_idx, scalars)
    d_out = torch.full((n, 32), 0xAA, dtype=torch.uint8, device=d_s.device)
    d_st = torch.full((n,), 99, dtype=torch.uint8, device=d_s.device)
    s = stream if stream is not None else torch.cuda.current_stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ks.dev_mul(n, d_idx, d_s, d_out, d_st, flags=flags)
    s.synchronize()
    return d_out.cpu().numpy(), d_st.cpu().numpy()


@pytest.mark.parametrize("flags", FLAGS)
def test_keyset_mul_key_and_scalar_classes(ctx, coracle, golden_records, flags):
    """Every key class against every scalar class (edges of the recoding, top bytes above 0x7f, all-0xff, random): host and
    device forms equal kb_point_mul_batch, and the oracle wherever the key decodes."""
    keys = _key_classes(golden_records, coracle)
    sc = _arr(scalar_classes())
    nk, ns = keys.shape[0], sc.shape[0]
    key_idx = np.repeat(np.arange(nk, dtype=np.uint32), ns)
    scalars = np.tile(sc, (nk, 1))
    pts = keys[key_idx]
    want, want_st = ctx.point_mul_batch(scalars, pts, flags)
    dec = np.array([coracle.point_decode_ok(k.tobytes()) for k in keys])
    assert (~dec).sum() >= 3 and (want_st == (~dec[key_idx]).astype(np.uint8)).all()
    ok = want_st == 0
    assert (want[ok] == coracle.mul_batch(scalars[ok], pts[ok], nthreads=8)).all()
    ks = ctx.keyset(keys)
    try:
        out, st = ks.mul_batch(key_idx, scalars, flags)
        assert (st == want_st).all() and (out == want).all(), np.nonzero((out != want).any(axis=1))[0][:10]
        out, st = _dev_mul(ks, key_idx, scalars, flags)
        assert (st == want_st).all() and (out == want).all(), np.nonzero((out != want).any(axis=1))[0][:10]
    finally:
        ks.close()


def test_keyset_mul_mostly_combless_keys(ctx, coracle, golden_records):
    """A batch in which most items use keys without a comb (weak, non-canonical, undecodable), shuffled among items of keys
    with one, so that the two paths of the kernel run side by side in every warp."""
    keys = _key_classes(golden_records, coracle)
    chk = ctx.point_check_batch(keys)   # bit 0 canonical, bit 1 small order, bit 2 decodes: a comb is built for 0b101
    combless = (chk & 7) != 5
    assert combless.sum() >= 10
    rng = np.random.default_rng(11)
    n = 6000
    pick = rng.random(n) < 0.8
    key_idx = np.where(pick, rng.choice(np.nonzero(combless)[0], n), rng.choice(np.nonzero(~combless)[0], n)).astype(np.uint32)
    scalars = np.frombuffer(xof_bytes("kyber-b200/test/keyset-mul/combless", 32 * n), dtype=np.uint8).reshape(n, 32).copy()
    ks = ctx.keyset(keys)
    try:
        for flags in FLAGS:
            want, want_st = ctx.point_mul_batch(scalars, keys[key_idx], flags)
            assert want_st.any() and not want_st.all()
            out, st = ks.mul_batch(key_idx, scalars, flags)
            assert (st == want_st).all() and (out == want).all()
            out, st = _dev_mul(ks, key_idx, scalars, flags)
            assert (st == want_st).all() and (out == want).all()
    finally:
        ks.close()


def test_keyset_mul_argument_errors(kb, ctx, golden_records):
    """key_idx >= nkeys: KBError on the host form, status 0xFF and 32 zero bytes for exactly those items on the device form;
    flags other than 0 / KB_FLAG_VARTIME: KBError on every form; n = 0 is accepted."""
    keys = _arr([r[1] for r in golden_records[:9]])
    n = 300
    rng = np.random.default_rng(4)
    key_idx = rng.integers(0, 9, size=n, dtype=np.uint32)
    scalars = np.frombuffer(xof_bytes("kyber-b200/test/keyset-mul/errors", 32 * n), dtype=np.uint8).reshape(n, 32).copy()
    want, want_st = ctx.point_mul_batch(scalars, keys[key_idx])
    ks = ctx.keyset(keys)
    try:
        bad = key_idx.copy()
        bad[5] = 9
        with pytest.raises(kb.KBError):
            ks.mul_batch(bad, scalars)
        bad[200] = 0xFFFFFFFF
        out, st = _dev_mul(ks, bad, scalars, 0)
        assert st[5] == st[200] == 0xFF and not out[[5, 200]].any()
        keep = np.ones(n, dtype=bool)
        keep[[5, 200]] = False
        assert (st[keep] == 0).all() and (out[keep] == want[keep]).all()
        for fl in (2, 3, 4, 0x80000000):
            with pytest.raises(kb.KBError):
                ks.mul_batch(key_idx, scalars, fl)
            with pytest.raises(kb.KBError):
                _dev_mul(ks, key_idx, scalars, fl)
        out, st = ks.mul_batch(key_idx, scalars)   # still usable
        assert (out == want).all() and (st == want_st).all()
        e = np.zeros(0, dtype=np.uint32)
        assert ks.mul_batch(e, np.zeros((0, 32), dtype=np.uint8))[0].shape == (0, 32)
        ks.dev_mul(0, None, None, None, None)
    finally:
        ks.close()


@pytest.mark.parametrize("flags", FLAGS)
def test_keyset_mul_large_batch(ctx, flags):
    """2^20 items under 1024 keys with random indices, device form on a non-default stream, against kb_dev_point_mul with
    points = keys[key_idx]; a sample against the C oracle is covered by the class test."""
    import torch

    n, nkeys = 1 << 20, 1024
    rng = np.random.default_rng(flags + 1)
    kseeds = np.frombuffer(xof_bytes("kyber-b200/test/keyset-mul/large-keys", 32 * nkeys), dtype=np.uint8).reshape(nkeys, 32).copy()
    keys = ctx.point_mul_base_batch(kseeds)
    key_idx = rng.integers(0, nkeys, size=n, dtype=np.uint32)
    scalars = np.frombuffer(xof_bytes(f"kyber-b200/test/keyset-mul/large/{flags}", 32 * n), dtype=np.uint8).reshape(n, 32).copy()
    d_pts, d_s = _to_dev(keys[key_idx], scalars)
    d_want = torch.empty((n, 32), dtype=torch.uint8, device=d_s.device)
    d_wst = torch.full((n,), 99, dtype=torch.uint8, device=d_s.device)
    ctx.dev_point_mul(n, d_s, d_pts, d_want, d_wst, flags)
    torch.cuda.synchronize()
    want, want_st = d_want.cpu().numpy(), d_wst.cpu().numpy()
    assert not want_st.any()
    ks = ctx.keyset(keys)
    try:
        out, st = _dev_mul(ks, key_idx, scalars, flags, stream=torch.cuda.Stream())
        assert not st.any() and (out == want).all(), np.nonzero((out != want).any(axis=1))[0][:10]
    finally:
        ks.close()


_LAYOUT = r"""
#define KB_HOST_EMU 1
#include <stddef.h>
#include "ctx.cuh"
int main() { printf("%zu %zu\n", offsetof(kb_ctx, slot), offsetof(kb_ctx, slot_bytes)); return 0; }
"""


def _scratch_slot0(ctx, tmp_path):
    """Bytes of the context's scratch slot 0 (where the host forms stage their scalars): the slot's device pointer and size
    read from the kb_ctx struct (offsets from a host build of csrc/ctx.cuh), copied with the driver API."""
    src = tmp_path / "layout.cpp"
    src.write_text(_LAYOUT)
    exe = tmp_path / "layout"
    subprocess.check_call(["g++", "-std=c++17", "-I/usr/local/cuda/include", "-I", os.path.join(ROOT, "kyber-rs_b200", "csrc"), "-o", str(exe), str(src)])
    off_slot, off_bytes = (int(x) for x in subprocess.check_output([str(exe)]).split())
    base = ctx.h.value
    ptr = ctypes.c_uint64.from_address(base + off_slot).value
    size = ctypes.c_size_t.from_address(base + off_bytes).value
    assert ptr and size
    cu = ctypes.CDLL("libcuda.so.1")
    buf = ctypes.create_string_buffer(size)
    assert cu.cuMemcpyDtoH_v2(buf, ctypes.c_uint64(ptr), ctypes.c_size_t(size)) == 0
    return buf.raw


def test_keyset_mul_scratch(ctx, golden_records, tmp_path):
    """The host form zeroes the scalars it staged unless KB_FLAG_VARTIME declares them public; kb_ctx_wipe between calls
    leaves the key set usable (its combs are not scratch)."""
    keys = _arr([r[1] for r in golden_records[:5]])
    n = 4096
    key_idx = (np.arange(n) % 5).astype(np.uint32)
    scalars = np.frombuffer(xof_bytes("kyber-b200/test/keyset-mul/scratch", 32 * n), dtype=np.uint8).reshape(n, 32).copy()
    want, _ = ctx.point_mul_batch(scalars, keys[key_idx])
    ks = ctx.keyset(keys)
    try:
        out, _ = ks.mul_batch(key_idx, scalars)
        assert (out == want).all()
        slot0 = _scratch_slot0(ctx, tmp_path)
        assert slot0[:32 * n] == bytes(32 * n)
        out, _ = ks.mul_batch(key_idx, scalars, 1)   # public scalars stay staged: the probe does see them
        assert (out == want).all()
        assert _scratch_slot0(ctx, tmp_path)[:32 * n] == scalars.tobytes()
        ctx.wipe()
        assert _scratch_slot0(ctx, tmp_path)[:32 * n] == bytes(32 * n)
        out, _ = ks.mul_batch(key_idx, scalars)
        assert (out == want).all()
        ctx.wipe()
        d_out, _ = _dev_mul(ks, key_idx, scalars, 0)
        assert (d_out == want).all()
    finally:
        ks.close()


@pytest.mark.parametrize("which", ["one", "all"])
def test_keyset_mul_multi_device(kb, ctx, golden_records, coracle, which):
    """MultiKeySet.mul_batch with the devices present (a batch that does not divide evenly) equals the single-device result;
    a bad index or flag is refused before any device starts."""
    import torch

    ngpu = torch.cuda.device_count()
    if which == "all" and ngpu < 2:
        pytest.skip("a single GPU is visible")
    devs = [0] if which == "one" else list(range(min(ngpu, 8)))
    keys = _key_classes(golden_records, coracle)
    n = 10007
    rng = np.random.default_rng(9)
    key_idx = rng.integers(0, keys.shape[0], size=n, dtype=np.uint32)
    scalars = np.frombuffer(xof_bytes("kyber-b200/test/keyset-mul/multi", 32 * n), dtype=np.uint8).reshape(n, 32).copy()
    ks = ctx.keyset(keys)
    m = kb.MultiContext(devs)
    mk = m.keyset(keys)
    try:
        for flags in FLAGS:
            want, want_st = ks.mul_batch(key_idx, scalars, flags)
            out, st = mk.mul_batch(key_idx, scalars, flags)
            assert (out == want).all() and (st == want_st).all()
        bad = key_idx.copy()
        bad[-1] = keys.shape[0]
        with pytest.raises(kb.KBError):
            mk.mul_batch(bad, scalars)
        with pytest.raises(kb.KBError):
            mk.mul_batch(key_idx, scalars, 2)
    finally:
        mk.close()
        m.close()
        ks.close()


def test_keyset_mul_from_plain_c(kb, ctx, golden_records, coracle, tmp_path):
    """tests/c/keyset_mul_check.c: create / kb_keyset_mul_batch (flags 0 and VARTIME) / destroy from plain C (gcc,
    -lkyber_b200), on a fixture whose expected bytes come from kb_point_mul_batch."""
    keys = _key_classes(golden_records, coracle)
    n = 3000
    rng = np.random.default_rng(21)
    key_idx = rng.integers(0, keys.shape[0], size=n, dtype=np.uint32)
    scalars = np.frombuffer(xof_bytes("kyber-b200/test/keyset-mul/c", 32 * n), dtype=np.uint8).reshape(n, 32).copy()
    want, want_st = ctx.point_mul_batch(scalars, keys[key_idx])
    fx = tmp_path / "fixture.bin"
    with open(fx, "wb") as f:
        f.write(np.array([n, keys.shape[0]], dtype=np.uint64).tobytes())
        for a in (keys, key_idx, scalars, want, want_st):
            f.write(np.ascontiguousarray(a).tobytes())
    exe = tmp_path / "keyset_mul_check"
    libdir = os.path.dirname(kb.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-O1", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "keyset_mul_check.c"),
                           "-L", libdir, "-lkyber_b200", "-Wl,-rpath," + libdir, "-o", str(exe)])
    r = subprocess.run([str(exe), str(fx)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "mismatches=0" in r.stdout
