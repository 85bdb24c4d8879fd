"""Batched share checks of a DKG round (dkgrlc.cuh) in the host emulation of the device math (tests/emu/emu_round_batched.cpp
compiles the same headers the kernels inline): the weights w_j, the share sums S_d and the torsion classes against Python
integers and the oracle's point arithmetic, at every residue of x mod 8.  CPU only."""
import ctypes
import hashlib
import os
import random
import subprocess

import pytest

from helpers import ROOT
from oracle import ed25519_bigint as O

L = O.L
PASS, FALLBACK = 0x100, 0x200


@pytest.fixture(scope="module")
def emu():
    d = os.path.join(ROOT, "tests", "emu")
    so = os.path.join(d, "_emu_round_batched.so")
    srcs = [os.path.join(d, "emu.cpp"), os.path.join(d, "emu_round_batched.cpp")] + [os.path.join(ROOT, "kyber-rs_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "kyber-rs_b200", "csrc")) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unused-function", "-o", so, os.path.join(d, "emu_round_batched.cpp")])
    E = ctypes.CDLL(so)
    sz = ctypes.c_size_t
    E.emu_rc_weights.argtypes = [sz, sz, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p]
    E.emu_rc_recode.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_int16)]
    E.emu_rc_torsion_mask.argtypes = [sz, ctypes.c_char_p]
    E.emu_rc_torsion_mask.restype = ctypes.c_uint32
    E.emu_rc_dealer.argtypes = [sz, sz, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, sz, ctypes.c_char_p]
    E.emu_rc_dealer.restype = ctypes.c_uint32
    return E


def _b(x: int) -> bytes:
    return x.to_bytes(32, "little")


def _torsion_points():
    """One point of each order 2, 4 and 8 (the oracle's small-order encodings)."""
    pts = [O.point_decode(k) for k in O.WEAK_KEYS]
    out = {}
    for p in pts:
        if p is None:
            continue
        for order in (2, 4, 8):
            if O._mul_int(order, p) == O.IDENTITY and all(O._mul_int(o, p) != O.IDENTITY for o in (1, 2, 4) if o < order):
                out.setdefault(order, p)
    # an order-8 point gives the orders 4 and 2 as its multiples
    t8 = out[8]
    out.setdefault(4, O._mul_int(2, t8))
    out.setdefault(2, O._mul_int(4, t8))
    return out


def _dealer(rnd, t, n, torsion=None, wrong=()):
    """Commitments (with torsion[j] added to C_j) and the honest shares s_i = f(x_i) mod L, except the indices in wrong."""
    coeffs = [rnd.randrange(L) for _ in range(t)]
    commits = [O.point_mul(_b(a)) for a in coeffs]
    for j, tp in (torsion or {}).items():
        commits[j] = O.point_add(commits[j], tp)
    shares = []
    for i in range(n):
        x = i + 1
        s = sum(a * pow(x, j, L) for j, a in enumerate(coeffs)) % L
        if i in wrong:
            s = (s + 1 + rnd.randrange(L - 1)) % L
        shares.append(_b(s))
    return commits, shares


def _exact_pattern(commits, shares):
    return [int(O.pubpoly_check(commits, i, s)) for i, s in enumerate(shares)]


def test_weights_match_python_integers(emu):
    """z_i = SHA-512(seed || i || 0^48)[:16] and w_j = sum_i z_i x_i^j mod L, for several n and t (chunks of 32 weights)."""
    rnd = random.Random(5)
    for n, t in ((1, 1), (8, 3), (37, 33), (64, 70)):
        seed = rnd.randbytes(32)
        z16, w32 = ctypes.create_string_buffer(16 * n), ctypes.create_string_buffer(32 * t)
        emu.emu_rc_weights(n, t, seed, z16, w32)
        z = [int.from_bytes(z16.raw[16 * i:16 * i + 16], "little") for i in range(n)]
        for i in range(n):
            want = hashlib.sha512(seed + i.to_bytes(8, "little") + bytes(24)).digest()[:16]
            assert z[i] == int.from_bytes(want, "little"), (n, i)
        for j in range(t):
            want = sum(z[i] * pow(i + 1, j, L) for i in range(n)) % L
            assert int.from_bytes(w32.raw[32 * j:32 * j + 32], "little") == want, (n, t, j)


def test_recode_radix256(emu):
    rnd = random.Random(6)
    vals = [0, 1, 127, 128, 129, 255, 256, L - 1, (1 << 253) - 1] + [rnd.randrange(L) for _ in range(200)]
    e = (ctypes.c_int16 * 32)()
    for v in vals:
        emu.emu_rc_recode(_b(v), e)
        assert all(-127 <= d <= 128 for d in e)
        assert sum(d * 256**k for k, d in enumerate(e)) == v


def test_torsion_mask_every_residue(emu):
    """The mask from the [L] images of A_even, A_odd, C_0, C_1, C_2 equals the torsion part of the exact eval(x) for every
    x mod 8: torsion of orders 2, 4, 8 on coefficients 0, 1, 2, 3, t - 1 and on even / odd pairs that cancel."""
    tor = _torsion_points()
    rnd = random.Random(7)
    cases = []
    for t in (1, 2, 3, 4, 5, 9):
        for order, tp in tor.items():
            for j in sorted({0, 1, 2, 3, t - 1}):
                if j < t:
                    cases.append((t, {j: tp}))
        if t >= 3:
            cases.append((t, {0: tor[8], 2: O.point_neg(tor[8])}))   # cancels for every x
            cases.append((t, {1: tor[4], 2: tor[2]}))
        if t >= 4:
            cases.append((t, {1: tor[8], 3: O.point_neg(tor[8])}))   # cancels for odd x only
    for t, tdict in cases:
        coeffs = [rnd.randrange(L) for _ in range(t)]
        commits = [O.point_mul(_b(a)) for a in coeffs]
        for j, tp in tdict.items():
            commits[j] = O.point_add(commits[j], tp)
        mask = emu.emu_rc_torsion_mask(t, b"".join(O.point_encode(c) for c in commits))
        for r in range(8):
            x = r if r else 8
            # torsion part of eval(x) = sum_j x^j tau_j
            acc = O.IDENTITY
            for j, tp in tdict.items():
                acc = O.point_add(acc, O._mul_int(x**j, tp))
            assert ((mask >> r) & 1) == int(acc == O.IDENTITY), (t, sorted(tdict), r)


@pytest.mark.parametrize("nch", [1, 3])
def test_dealer_state_against_exact_checks(emu, nch):
    """The whole per-dealer decision: honest dealers pass with the mask of their exact verdicts (torsion included), a dealer
    with one wrong share or a share with byte 31 > 127 falls back, S_d = sum z_i s_i mod L."""
    tor = _torsion_points()
    rnd = random.Random(8 + nch)
    n = 16   # every residue of x mod 8 twice
    for t, tdict, wrong in ((1, None, ()), (4, None, ()), (5, {0: tor[8]}, ()), (5, {1: tor[4], 4: tor[2]}, ()), (3, {2: tor[8]}, ()),
                            (4, None, (3,)), (6, {1: tor[8]}, (0,)), (40, None, ())):
        commits, shares = _dealer(rnd, t, n, tdict, wrong)
        cb = b"".join(O.point_encode(c) for c in commits)
        seed = rnd.randbytes(32)
        s_out = ctypes.create_string_buffer(32)
        state = emu.emu_rc_dealer(n, t, cb, b"".join(shares), seed, nch, s_out)
        z16, w32 = ctypes.create_string_buffer(16 * n), ctypes.create_string_buffer(32 * t)
        emu.emu_rc_weights(n, t, seed, z16, w32)
        z = [int.from_bytes(z16.raw[16 * i:16 * i + 16], "little") for i in range(n)]
        assert int.from_bytes(s_out.raw, "little") == sum(zi * int.from_bytes(s, "little") for zi, s in zip(z, shares)) % L
        exact = _exact_pattern(commits, shares)
        if wrong:
            assert state == FALLBACK, (t, wrong)
            continue
        assert state & PASS, (t, tdict)
        assert [(state >> ((i + 1) & 7)) & 1 for i in range(n)] == exact, (t, tdict)
    # honest shares given as s + L stay on the fast path; byte 31 > 127 falls back
    commits, shares = _dealer(rnd, 3, n)
    cb = b"".join(O.point_encode(c) for c in commits)
    plus_l = [_b(int.from_bytes(s, "little") + L) for s in shares]
    s_out = ctypes.create_string_buffer(32)
    assert emu.emu_rc_dealer(n, 3, cb, b"".join(plus_l), rnd.randbytes(32), nch, s_out) == PASS | 0xFF
    high = list(shares)
    high[5] = _b(int.from_bytes(high[5], "little") + (1 << 255))
    assert emu.emu_rc_dealer(n, 3, cb, b"".join(high), rnd.randbytes(32), nch, s_out) == FALLBACK
