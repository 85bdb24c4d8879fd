"""The closed-form MSM reference (tests/msm_reference.py) against the oracles, and the host emulation of the Pippenger
stage bodies (tests/emu/emu.cpp) against the closed form at every window width and bucket grouping the driver uses.
CPU only; the GPU counterpart is tests/test_gpu_msm_reference.py."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import msm_reference as R
from helpers import ROOT
from oracle import ed25519_bigint as O

L = O.L


@pytest.fixture(scope="module")
def emu():
    d = os.path.join(ROOT, "tests", "emu")
    so = os.path.join(d, "_emu.so")
    srcs = [os.path.join(d, "emu.cpp")] + [os.path.join(ROOT, "kyber-rs_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "kyber-rs_b200", "csrc")) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unused-function", "-o", so, os.path.join(d, "emu.cpp")])
    E = ctypes.CDLL(so)
    E.emu_msm_plan.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    return E


def emu_msm(emu, s, p, c=0, groups=0):
    s, p = np.ascontiguousarray(s, dtype=np.uint8), np.ascontiguousarray(p, dtype=np.uint8)
    out = ctypes.create_string_buffer(32)
    bad = emu.emu_msm_plan(out, s.shape[0], s.ctypes.data, p.ctypes.data, c, 0, groups)
    return out.raw, bad


@pytest.fixture(scope="module")
def pts1024(coracle):
    return R.oracle_points(1024, 11, coracle)


def test_effective_rule_matches_oracle():
    """The vectorised effective-scalar rule, and its one-integer form, are the reference's on random raw scalars,
    every edge scalar and the structured families."""
    rng = np.random.default_rng(3)
    s = np.concatenate([rng.integers(0, 256, size=(3000, 32), dtype=np.uint8), R.EDGES, R.carry_chain(64, 1, 13), R.small(64, 1, 16)])
    s[:256, 31] = np.arange(256, dtype=np.uint8)                     # every top byte
    mag, neg = R.effective(s)
    for k, row in enumerate(s):
        want = O.scalar_effective(row.tobytes())
        got = sum(int(mag[j, k]) << (16 * j) for j in range(16)) - (int(neg[k]) << 252)
        assert got == want == R.effective_int(row.tobytes()), row.tobytes().hex()
        assert want % 8 == int.from_bytes(row.tobytes(), "little") % 8
    assert neg.any() and (~neg).any()


@pytest.mark.parametrize("family", sorted(R.FAMILIES))
def test_closed_form_matches_oracle_small(coracle, family):
    """n <= 64 with torsion components, repeated points and P, -P pairs: the closed form is the oracle's MSM."""
    n = 64
    r, t = R.point_logs(n, 5)
    r[10:14], t[10:14] = r[3], t[3]                                  # the same point four more times
    neg_r = R.to_bytes([(L - v) % L for v in R.to_ints(r[20:26])])
    r[26:32], t[26:32] = neg_r, (8 - t[20:26].astype(np.int64)) % 8   # -P of points 20..25
    pts = np.frombuffer(b"".join(O.point_encode(O.point_add(O._mul_int(R.to_ints(r[i:i + 1])[0], O.BASE), O._mul_int(int(t[i]), O.point_decode(R.T8)))) for i in range(n)), dtype=np.uint8).reshape(n, 32)
    assert pts[26:32].tobytes() == b"".join(O.point_encode(O.point_neg(O.point_decode(p.tobytes()))) for p in pts[20:26])
    for c in (4, 9):
        s = R.FAMILIES[family](n, 7, c)
        want = R.expected(s, r, t)
        assert want == coracle.msm(s, pts)
        if c == 4:
            assert want == O.point_encode(O.msm([x.tobytes() for x in s], [O.point_decode(p.tobytes()) for p in pts]))


def test_closed_form_every_edge_scalar(coracle):
    """Each edge scalar alone, on a point with a torsion component, and all of them in one MSM."""
    m = R.EDGES.shape[0]
    r, t = R.point_logs(m, 9)
    t[:] = np.arange(m) % 7 + 1
    base = coracle.mul_base_batch(r, nthreads=8)
    pts = np.frombuffer(b"".join(coracle.point_add(b.tobytes(), R.TORSION[k].tobytes()) for b, k in zip(base, t)), dtype=np.uint8).reshape(m, 32)
    for i in range(m):
        assert R.expected(R.EDGES[i:i + 1], r[i:i + 1], t[i:i + 1]) == coracle.mul(R.EDGES[i].tobytes(), pts[i].tobytes())
    assert R.expected(R.EDGES, r, t) == coracle.msm(R.EDGES, pts)


def test_closed_form_large_block_sum(coracle, pts1024):
    """More rows than one float64 block of the exact dot product: tiling 1024 points 300 times multiplies the sum."""
    pts, r, t = pts1024
    s = R.uniform(1024, 2)
    want = coracle.msm(s, pts)
    reps = 300                                                        # 307 200 rows > 2^18
    got = R.expected(np.tile(s, (reps, 1)), np.tile(r, (reps, 1)), np.tile(t, reps))
    assert got == coracle.mul(reps.to_bytes(32, "little"), want)


@pytest.mark.parametrize("c", range(4, 17))
def test_emulated_stages_every_window_width(emu, pts1024, c):
    """The stage bodies with the device's window width and bucket grouping for c = 4..16, against the closed form."""
    pts, r, t = pts1024
    n = 1024 if c <= 12 else 512
    for family in ("uniform", "carry", "edges", "reduced"):
        s = R.FAMILIES[family](n, 100 + c, c)
        got, bad = emu_msm(emu, s, pts[:n], c)
        assert bad == 0 and got == R.expected(s, r[:n], t[:n]), (family, c)


@pytest.mark.parametrize("c,groups", [(14, 32), (14, 33), (14, 3000), (16, 33), (16, 3000), (15, 16384), (13, 3000)])
def test_emulated_stages_bucket_groups(emu, pts1024, c, groups):
    """KB_MSM_GROUPS settings that give several groups per thread in the window fold and group sizes that do not
    divide the window (33, 3000), and one clipped to the bucket count (16384 at c = 15)."""
    pts, r, t = pts1024
    n = 512
    for family in ("uniform", "carry"):
        s = R.FAMILIES[family](n, 200 + groups, c)
        got, bad = emu_msm(emu, s, pts[:n], c, groups)
        assert bad == 0 and got == R.expected(s, r[:n], t[:n]), (family, c, groups)


def test_emulated_stages_skewed_families(emu, pts1024):
    """One bucket per window (all scalars equal), mostly zero scalars and window-0-only scalars, at the size rule."""
    pts, r, t = pts1024
    for family in ("equal", "sparse", "small"):
        for c in (0, 6, 11):
            s = R.FAMILIES[family](1024, 300 + c, c or 7)
            got, bad = emu_msm(emu, s, pts, c)
            assert bad == 0 and got == R.expected(s, r, t), (family, c)
