"""The short-wrap field bodies of the verify kernels (fe.cuh fe_sw) and the exact redo behind them.

k_verify_half_main ends every field operation of its table build and loop with a carry that stops at word 1; a carry or
borrow out of word 1 is counted in a per-thread `ovf` instead of rippling on, and a thread whose count is not 0 redoes its
record with the exact bodies.  Checked here:
  * the invariant, on the host build and on the device (tests/gpu_math/short_wrap_harness.cu): ovf == 0 implies the raw
    output equals the exact body's, on random operands and on operands built to carry out of word 1;
  * that honest signatures never raise ovf (the redo costs nothing in practice), on the host emulation of the kernel;
  * that the redo is exact: with KB_VERIFY_FORCE_REDO every (or every k-th) thread takes it, and every status equals the
    unforced run's and the reference's (host emulation and B200)."""
import ctypes
import functools
import importlib
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

from helpers import FE_EDGE, P_FIELD, ROOT, make_mixed_order_sigs, make_sig_batch, pack_batch

P = P_FIELD
M = 2**256
CSRC = os.path.join(ROOT, "kyber-rs_b200", "csrc")
HARNESS_SRC = os.path.join(ROOT, "tests", "gpu_math", "short_wrap_harness.cu")
GPU_DEFINES = {"gpu-rows": [], "gpu-rip": ["-DKB_FE_MUL_RIP", "-DKB_FE_SQ_RIP", "-DKB_FE_SUBMASK"]}
OPS = {name: i for i, name in enumerate(["mul", "sq", "add", "sub", "dbl", "neg", "reduce512"])}
BACKENDS = [pytest.param("emu", id="emu"), pytest.param("gpu-rows", id="gpu-rows", marks=pytest.mark.gpu), pytest.param("gpu-rip", id="gpu-rip", marks=pytest.mark.gpu)]
NRAND = 4096


def find_nvcc():
    nvcc = shutil.which("nvcc")
    if nvcc is None and os.path.exists("/usr/local/cuda/bin/nvcc"):
        nvcc = "/usr/local/cuda/bin/nvcc"
    return nvcc


def build_harness(backend, out):
    if backend == "emu":
        cmd = ["g++", "-x", "c++", "-DKB_HOST_EMU", "-O2", "-std=c++17", "-fPIC", "-shared"]
    else:
        nvcc = find_nvcc()
        assert nvcc is not None, "nvcc not found: the device build of the short-wrap harness needs the CUDA toolkit"
        cmd = [nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared", "-diag-suppress", "177"] + GPU_DEFINES[backend]
    cmd += ["-I", CSRC, "-o", str(out), HARNESS_SRC]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, f"building the {backend} short-wrap harness failed:\n{' '.join(cmd)}\n{r.stdout}{r.stderr}"
    lib = ctypes.CDLL(str(out))
    lib.fe_sw_batch.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    return lib


@pytest.fixture(scope="module")
def harness_cache(tmp_path_factory):
    d = tmp_path_factory.mktemp("short_wrap_harness")
    return functools.lru_cache(maxsize=None)(lambda backend: build_harness(backend, d / f"short_wrap_{backend}.so"))


def run(lib, op, exact, a, b):
    a = np.ascontiguousarray(a, dtype=np.uint32)
    b = np.ascontiguousarray(b, dtype=np.uint32)
    out = np.empty_like(a)
    ovf = np.empty(a.shape[0], dtype=np.uint32)
    rc = lib.fe_sw_batch(OPS[op], exact, a.shape[0], a.ctypes.data, b.ctypes.data, out.ctypes.data, ovf.ctypes.data)
    assert rc == 0, f"fe_sw_batch({op}) returned {rc}"
    return out, ovf


def words(xs):
    return np.array([[(x >> (32 * k)) & 0xFFFFFFFF for k in range(8)] for x in xs], dtype=np.uint32).reshape(-1, 8)


def ints(w):
    return [sum(int(r[k]) << (32 * k) for k in range(8)) for r in w]


def operands(op, rnd):
    """(a, b, edge) for `op`: random 256-bit operands, the edge values of the field tests, and operands built so that the
    short wrap carries (or borrows) out of word 1 — `edge` marks those, which must raise ovf."""
    a, b, edge = [], [], []
    for _ in range(NRAND):
        a.append(rnd.getrandbits(256)); b.append(rnd.getrandbits(256)); edge.append(False)
    for x in FE_EDGE:
        for y in FE_EDGE[::3]:
            a.append(x % M); b.append(y % M); edge.append(False)
    for x in [P + k for k in range(0, 40)] + [M - 1 - k for k in range(40)]:
        a.append(x); b.append(rnd.getrandbits(256)); edge.append(False)
    for _ in range(512):
        lo = (0xFFFFFFFF << 32)
        if op == "add":
            # f + g = 2^256 + T with word 1 of T all ones and word 0 within 38 of the top: the wrap adds 38 and carries out of word 1
            t = (rnd.getrandbits(192) << 64) | lo | (0xFFFFFFFF - rnd.randrange(38))
            s = M + t
            f = rnd.randrange(s - M + 1, M)
            a.append(f); b.append(s - f); edge.append(True)
        elif op == "dbl":
            t = (rnd.getrandbits(192) << 64) | lo | (0xFFFFFFFE - 2 * rnd.randrange(19))
            a.append((M + t) // 2); b.append(0); edge.append(True)
        elif op in ("sub", "neg"):
            # f - g = T - 2^256 with T < 38 in words 0..1: the wrap subtracts 38 and borrows out of word 1
            t = (rnd.getrandbits(192) << 64) | rnd.randrange(38)
            if op == "neg":
                if t == 0:
                    continue
                a.append(M - t); b.append(0); edge.append(True)   # 0 - (2^256 - t) = t - 2^256
            else:
                g = rnd.randrange(M - t, M)
                a.append(t + g - M); b.append(g); edge.append(True)
        elif op == "reduce512":
            # low half: word 0 within 1444 of the top, word 1 all ones; high half: only word 7, so that the fold leaves words
            # 0 and 1 alone and its top word is 1 .. 37: the final wrap adds 38 * top and carries out of word 1
            x = rnd.randrange(2**32 // 38 + 1, 2**32)
            top = (38 * x) >> 32
            lo_half = (rnd.getrandbits(192) << 64) | lo | (2**32 - 1 - rnd.randrange(38 * top))
            a.append(lo_half); b.append(x << 224); edge.append(True)
    return words(a), words(b), np.array(edge)


def reference(op, x, y):
    if op == "mul":
        return x * y % P
    if op == "sq":
        return x * x % P
    if op == "add":
        return (x + y) % P
    if op == "sub":
        return (x - y) % P
    if op == "dbl":
        return 2 * x % P
    if op == "neg":
        return -x % P
    return (x + (y << 256)) % P


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("op", list(OPS))
def test_short_wrap_equals_exact_unless_flagged(harness_cache, backend, op):
    """ovf == 0 implies the raw output equals the exact body's; the built edge operands raise ovf; every exact output is
    the big-integer result mod p.  The device builds agree with the host build bit for bit (outputs and counters)."""
    lib = harness_cache(backend)
    a, b, edge = operands(op, random.Random(f"short-wrap/{op}"))
    ex, ex_ovf = run(lib, op, 1, a, b)
    sw, ovf = run(lib, op, 0, a, b)
    assert not ex_ovf.any()
    same = (ex == sw).all(axis=1)
    assert same[ovf == 0].all(), f"{op}: short-wrap output differs from the exact one without raising ovf"
    assert (ovf[edge] != 0).all(), f"{op}: an operand built to carry out of word 1 did not raise ovf"
    for x, y, r in zip(ints(a), ints(b), ints(ex)):
        assert r % P == reference(op, x, y)
    if backend != "emu":
        h_sw, h_ovf = run(harness_cache("emu"), op, 0, a, b)
        h_ex, _ = run(harness_cache("emu"), op, 1, a, b)
        assert (h_sw == sw).all() and (h_ovf == ovf).all() and (h_ex == ex).all()


# ---- the verifier on the host emulation --------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu_sw():
    d = os.path.join(ROOT, "tests", "emu")
    so = os.path.join(d, "_emu_short_wrap.so")
    srcs = [os.path.join(d, "emu.cpp"), os.path.join(d, "emu_short_wrap.cpp")] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unused-function", "-o", so, os.path.join(d, "emu_short_wrap.cpp")])
    E = ctypes.CDLL(so)
    E.emu_sig_verify_half_sw.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    return E


def verify_sw(E, sch, pk, msg, sig, min_windows=0, force=0):
    ovf = ctypes.c_uint32()
    st = E.emu_sig_verify_half_sw(sch, pk, msg, len(msg), sig, min_windows, force, ctypes.addressof(ovf))
    return st, ovf.value


def test_honest_signatures_never_raise_ovf(emu_sw, golden_records):
    """Every golden signature, under both schemes, through the emulated short-wrap table build and loop of k_verify_half_main
    (a quarter of them with the loop padded to 64 pairs, as a short lane in a block of long ones runs it): no thread raises
    ovf, so the exact redo never runs on honest input, and every status is 0."""
    lanes = flagged = 0
    for k, (_, pk, sig, msg) in enumerate(golden_records):
        for sch in (0, 1):
            # every fourth one with a 64-pair loop: the leading pairs of a lane shorter than its block's loop are zero
            st, ovf = verify_sw(emu_sw, sch, pk, msg, sig, 64 if k % 4 == 0 else 0)
            assert st == 0
            lanes += 1
            flagged += ovf != 0
    print(f"short-wrap counters raised: {flagged} of {lanes} verifications")
    assert flagged == 0


def test_forced_redo_is_exact_on_host(emu_sw, coracle, golden_records):
    """With the counter forced to 1 the exact redo computes every status; it equals the unforced one and the reference's,
    for every rejection class, mixed-order keys and forced 64-window loops."""
    pks, msgs, sigs = make_sig_batch(golden_records[1:256:3], 24 * 4, bad_every=1)
    good, bad = make_mixed_order_sigs(6)
    items = list(zip(pks, msgs, sigs)) + good + bad
    seen = set()
    for k, (pk, msg, sig) in enumerate(items):
        for sch in (0, 1):
            want = coracle.schnorr_verify(pk, msg, sig) if sch else coracle.eddsa_verify(pk, msg, sig)
            mw = (0, 64)[k % 2]
            st0, _ = verify_sw(emu_sw, sch, pk, msg, sig, mw, 0)
            st1, forced = verify_sw(emu_sw, sch, pk, msg, sig, mw, 1)
            assert st0 == st1 == want
            assert forced >= 1
            seen.add(want)
    assert seen == {0, 2, 3, 4, 5, 6, 7, 8}


# ---- the kernels on the B200 -----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


def _ctx(kb, env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return kb.Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


@pytest.mark.gpu
@pytest.mark.parametrize("schnorr", [False, True])
def test_forced_redo_matches_unforced_on_gpu(kb, coracle, golden_records, schnorr):
    """A 2^16 batch (every rejection class, mixed-order keys) through k_verify_half_main with the exact
    redo forced on every thread and on every third, also with 64-window loops: every status equals the unforced run's and
    the reference's."""
    n = 2**16
    pks, msgs, sigs = make_sig_batch(golden_records, n - 64, bad_every=3)
    good, bad = make_mixed_order_sigs(32)
    for pk, msg, sig in good + bad:
        pks.append(pk); msgs.append(msg); sigs.append(sig)
    pk, flat, off, sg = pack_batch(pks, msgs, sigs)
    want = coracle.verify_batch(pk, flat, off, sg, nthreads=8, schnorr=schnorr)
    assert set(np.unique(want)) == {0, 2, 3, 4, 5, 6, 7, 8}
    for env in ({}, {"KB_VERIFY_FORCE_REDO": "1"}, {"KB_VERIFY_FORCE_REDO": "3"},
                {"KB_VERIFY_FORCE_REDO": "1", "KB_VERIFY_MIN_WINDOWS": "64"}, {"KB_VERIFY_FORCE_REDO": "5", "KB_VERIFY_SORT": "0"}):
        c = _ctx(kb, env)
        try:
            got = c.verify_batch(pk, flat, off, sg, schnorr=schnorr)
        finally:
            c.close()
        assert (got == want).all(), env
