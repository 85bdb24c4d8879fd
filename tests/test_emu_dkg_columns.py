"""Share checks of a verifier range (dkgcol.cuh) in the host emulation of the device math (tests/emu/emu_dkg_columns.cpp
compiles the same headers the kernels inline): the exponents x^j mod 8L and their digits against Python integers, and the
column evaluation sum_j e_j C_j against the oracle's Horner at x for commitments with torsion.  CPU only."""
import ctypes
import os
import random
import subprocess

import pytest

from helpers import ROOT
from oracle import ed25519_bigint as O

L = O.L
W = 33   # KB_COL_WINDOWS


@pytest.fixture(scope="module")
def emu():
    d = os.path.join(ROOT, "tests", "emu")
    so = os.path.join(d, "_emu_dkg_columns.so")
    srcs = [os.path.join(d, "emu.cpp"), os.path.join(d, "emu_dkg_columns.cpp")] + [os.path.join(ROOT, "kyber-rs_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "kyber-rs_b200", "csrc")) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unused-function", "-o", so, os.path.join(d, "emu_dkg_columns.cpp")])
    E = ctypes.CDLL(so)
    sz = ctypes.c_size_t
    E.emu_col_exponents.argtypes = [ctypes.c_uint64, sz, ctypes.c_char_p, ctypes.POINTER(ctypes.c_int16)]
    E.emu_col_recode.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_int16)]
    E.emu_col_eval.argtypes = [ctypes.c_char_p, ctypes.c_char_p, sz, ctypes.c_uint64, sz]
    E.emu_col_check.argtypes = [ctypes.c_char_p, sz, ctypes.c_uint64, ctypes.c_char_p, sz]
    return E


def _b(x: int) -> bytes:
    return x.to_bytes(32, "little")


def _digits_ok(d, v):
    assert all(-127 <= x <= 128 for x in d), v
    assert d[W - 1] in (0, 1), v
    assert sum(x * 256**k for k, x in enumerate(d)) == v, v


def test_exponents_and_digits_reconstruct(emu):
    """e_j = x^j mod 8L exactly, for x of every residue mod 8, x near 2^32 and t over several chunks of 32 exponents."""
    xs = list(range(1, 17)) + [1023, 1024, 1025, (1 << 32) - 1, 1 << 32]
    for x in xs:
        t = 70
        e32 = ctypes.create_string_buffer(32 * t)
        dig = (ctypes.c_int16 * (W * t))()
        emu.emu_col_exponents(x, t, e32, dig)
        for j in range(t):
            e = int.from_bytes(e32.raw[32 * j:32 * j + 32], "little")
            assert e == pow(x, j, 8 * L), (x, j)
            _digits_ok(list(dig[W * j:W * j + W]), e)


def test_recode_edges(emu):
    rnd = random.Random(11)
    vals = [0, 1, 128, 129, L - 1, L, 7 * L, 8 * L - 1, (1 << 255) - 1, 1 << 255, (1 << 255) + (1 << 127), 8 * L - 256]
    vals += [rnd.randrange(8 * L) for _ in range(300)]
    d = (ctypes.c_int16 * W)()
    for v in vals:
        emu.emu_col_recode(_b(v), d)
        _digits_ok(list(d), v)


def _torsion_points():
    pts = [O.point_decode(k) for k in O.WEAK_KEYS]
    out = {}
    for p in pts:
        if p is None:
            continue
        for order in (2, 4, 8):
            if O._mul_int(order, p) == O.IDENTITY and all(O._mul_int(o, p) != O.IDENTITY for o in (1, 2, 4) if o < order):
                out.setdefault(order, p)
    t8 = out[8]
    out.setdefault(4, O._mul_int(2, t8))
    out.setdefault(2, O._mul_int(4, t8))
    return out


@pytest.mark.parametrize("nch", [1, 2])
def test_column_eval_equals_horner_with_torsion(emu, nch):
    """sum_j (x^j mod 8L) C_j equals PubPoly::eval's Horner at the exact x: torsion of orders 2, 4, 8 on coefficients 0, 1, 2
    and t - 1, x of every residue mod 8 and a 32-bit x."""
    tor = _torsion_points()
    rnd = random.Random(12 + nch)
    for t in (1, 2, 3, 5, 43):
        coeffs = [rnd.randrange(L) for _ in range(t)]
        base = [O.point_mul(_b(a)) for a in coeffs]
        for order, tp in sorted(tor.items()):
            for j in sorted({0, 1, 2, t - 1}):
                if j >= t:
                    continue
                commits = list(base)
                commits[j] = O.point_add(commits[j], tp)
                cb = b"".join(O.point_encode(c) for c in commits)
                for x in list(range(1, 9)) + [(1 << 32) - 3]:
                    out = ctypes.create_string_buffer(32)
                    assert emu.emu_col_eval(out, cb, t, x, nch) == 1
                    assert out.raw == O.point_encode(O.pubpoly_eval(commits, x - 1)), (t, order, j, x)


def test_column_check_verdicts(emu):
    """The per-(column, dealer) verdict against the oracle's PubPoly::check: honest shares, s + L, byte 31 > 127, a wrong
    share, a torsion dealer; an undecodable commitment gives 0."""
    tor = _torsion_points()
    rnd = random.Random(13)
    t = 5
    coeffs = [rnd.randrange(L) for _ in range(t)]
    for tdict in ({}, {1: tor[8]}, {0: tor[4], 4: tor[2]}):
        commits = [O.point_mul(_b(a)) for a in coeffs]
        for j, tp in tdict.items():
            commits[j] = O.point_add(commits[j], tp)
        cb = b"".join(O.point_encode(c) for c in commits)
        for i in (0, 1, 2, 3, 4, 5, 6, 7, 1000):
            s = sum(a * pow(i + 1, j, L) for j, a in enumerate(coeffs)) % L
            for share in (_b(s), _b(s + L), _b(s + (1 << 255)), _b((s + 1) % L)):
                want = int(O.pubpoly_check(commits, i, share))
                assert emu.emu_col_check(cb, t, i + 1, share, 1) == want, (tdict, i, share.hex())
    bad = bytearray(b"".join(O.point_encode(O.point_mul(_b(a))) for a in coeffs))
    bad[32 * 2:32 * 3] = b"\x02" + b"\x00" * 30 + b"\x80"   # not on the curve
    assert O.point_decode(bytes(bad[64:96])) is None
    assert emu.emu_col_check(bytes(bad), t, 1, _b(0), 1) == 0
