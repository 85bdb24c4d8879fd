"""Keyed scalar multiplication (kb_keyset_mul_*) in the host emulation of the device math (tests/emu/emu_keyset_mul.cpp compiles
the same ops.cuh the kernels inline): the 64-window comb over a key's comb against the big-int oracle's Point::mul(s, Some(A)),
and the whole item against the emulated k_mul, for every scalar class that matters to the recoding.  CPU only."""
import ctypes
import os
import random
import subprocess

import pytest

from helpers import NONCANONICAL, ROOT, WEAK_KEYS, _off_curve
from oracle import ed25519_bigint as O

L = O.L


@pytest.fixture(scope="module")
def emu():
    d = os.path.join(ROOT, "tests", "emu")
    so = os.path.join(d, "_emu_keyset_mul.so")
    srcs = [os.path.join(d, "emu.cpp"), os.path.join(d, "emu_keyset_mul.cpp")] + [os.path.join(ROOT, "kyber-rs_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "kyber-rs_b200", "csrc")) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unused-function", "-o", so, os.path.join(d, "emu_keyset_mul.cpp")])
    E = ctypes.CDLL(so)
    E.emu_keyset_mul.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]
    E.emu_mul.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]
    return E


def _b(x: int) -> bytes:
    return x.to_bytes(32, "little")


def scalar_classes():
    """Edge scalars of the signed radix-16 recoding (sc_recode16), then 200 random ones.  A top byte above 0x7f makes the
    top digit 9..16, which the reference's table select turns into the identity: e[63] is zeroed."""
    rnd = random.Random(31)
    out = [_b(v) for v in (0, 1, 15, 16, L - 1, L, L + 1, 1 << 252, 8 * L - 1, (1 << 255) - 1)]
    for top in (0x7F, 0x80, 0x88, 0x8F, 0xF0, 0xFF):
        out.append(rnd.randbytes(31) + bytes([top]))
        out.append(b"\x00" * 31 + bytes([top]))
    out.append(b"\xff" * 32)
    out += [rnd.randbytes(32) for _ in range(200)]
    return out


def _torsion_key(pk, k):
    """A valid key plus k times a point of order 8: a key with a comb, of order 8L."""
    t8 = O.point_decode(O.WEAK_KEYS[2])
    return O.point_encode(O.point_add(O.point_decode(pk), O._mul_int(k, t8)))


def noncanonical_keys(coracle):
    """Encodings of y = p + t (t < 19, both signs of x) that decode: keys that are not canonical, some of small order."""
    cands = [bytes([0xED + t]) + b"\xff" * 30 + bytes([0x7F | sgn]) for t in range(19) for sgn in (0, 0x80)]
    out = [k for k in cands if coracle.point_decode_ok(k)]
    assert len(out) >= 4
    return out


def test_keyset_comb_mul_matches_oracle(emu, golden_records):
    """ge_keyset_mul<true> and <false> over the key comb equal the oracle's s*A, for a valid key and keys with a small-order
    component (exact multiples: 8L - 1 and scalars >= 2^255 are not reduced)."""
    keys = [golden_records[0][1], _torsion_key(golden_records[3][1], 1), _torsion_key(golden_records[5][1], 4)]
    scalars = scalar_classes()
    out = ctypes.create_string_buffer(32)
    for pk in keys:
        A = O.point_decode(pk)
        assert not O.point_has_small_order(A)
        for s in scalars:
            want = O.point_encode(O.point_mul(s, A))
            for ct in (1, 0):
                for direct in (1, 0):
                    assert emu.emu_keyset_mul(out, pk, s, ct, direct) == 0
                    assert out.raw == want, (pk.hex(), s.hex(), ct, direct)


def test_keyset_mul_item_equals_general_path(emu, coracle, golden_records):
    """The item as k_keyset_mul composes it equals the emulated k_mul byte for byte and status for status, for keys that have
    a comb and for every kind of key that has none: the weak keys, non-canonical encodings that decode, encodings in the
    is_canonical quirk range, and encodings that do not decode (identity, status 1)."""
    rnd = random.Random(7)
    keys = [golden_records[1][1], _torsion_key(golden_records[2][1], 2)] + WEAK_KEYS + noncanonical_keys(coracle)
    keys += [bytes([0x20]) + b"\xff" * 30 + b"\x7f", bytes([0x20]) + b"\xff" * 30 + b"\xff", NONCANONICAL, _off_curve(5), _off_curve(6)]
    decodes = [coracle.point_decode_ok(k) for k in keys]
    assert decodes.count(False) >= 2
    scalars = scalar_classes()[:22] + [rnd.randbytes(32) for _ in range(20)]
    got, ref = ctypes.create_string_buffer(32), ctypes.create_string_buffer(32)
    for pk, ok in zip(keys, decodes):
        for s in scalars:
            for ct in (1, 0):
                st = emu.emu_keyset_mul(got, pk, s, ct, 0)
                assert st == (0 if ok else 1)
                assert emu.emu_mul(ref, s, pk, ct) == int(ok)
                if ok:
                    assert got.raw == ref.raw, (pk.hex(), s.hex(), ct)
                    assert got.raw == O.point_encode(O.point_mul(s, O.point_decode(pk)))
                else:
                    assert got.raw == O.point_encode(O.IDENTITY)
