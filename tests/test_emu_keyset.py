"""Key sets (verification under registered public keys) in the host emulation of the device math
(tests/emu/emu_keyset.cpp compiles the same ops.cuh the kernels inline): the per-key comb against the big-int oracle, and the keyed verifier
against the reference's statuses.  CPU only."""
import ctypes
import os
import random
import subprocess

import pytest

from helpers import ROOT, WEAK_KEYS, make_mixed_order_sigs, mutate_signature
from oracle import ed25519_bigint as O

P = O.P
KEY_BITS, KEY_POS, KEY_HALF = 8, 32, 128   # ops.cuh KB_KEY_BITS / KB_KEY_POS / KB_KEY_HALF
F_AC, F_AS, F_AOK = 8, 16, 32              # ops.cuh KB_F_AC / KB_F_AS / KB_F_AOK


@pytest.fixture(scope="module")
def emu():
    d = os.path.join(ROOT, "tests", "emu")
    so = os.path.join(d, "_emu_keyset.so")
    srcs = [os.path.join(d, "emu.cpp"), os.path.join(d, "emu_keyset.cpp")] + [os.path.join(ROOT, "kyber-rs_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "kyber-rs_b200", "csrc")) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unused-function", "-o", so, os.path.join(d, "emu_keyset.cpp")])
    E = ctypes.CDLL(so)
    E.emu_keyset_row.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]
    E.emu_keyset_verify.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint64, ctypes.c_char_p]
    return E


def _affine_entry(pt):
    """(y+x, y-x, 2dxy) of an oracle point as the three canonical 32-byte fields of a comb entry."""
    x, y = pt
    return b"".join(v.to_bytes(32, "little") for v in ((y + x) % P, (y - x) % P, 2 * O.D * x * y % P))


def _torsion_key(rec_pk, k):
    """A valid key plus a point of order 8 (or 4, 2): passes the small-order filter, has order 8L."""
    t8 = O.point_decode(O.WEAK_KEYS[2])
    return O.point_encode(O.point_add(O.point_decode(rec_pk), O._mul_int(k, t8)))


def test_key_comb_entries(emu, coracle, golden_records):
    """kt[p][j] = (j+1) * 2^(8p) * A as exact integer multiples — for p = 31 the multiplier exceeds L, which matters for
    keys with a torsion component (order 8L) — for ordinary keys and torsion-carrying ones."""
    rnd = random.Random(17)
    keys = [golden_records[0][1], golden_records[9][1], _torsion_key(golden_records[3][1], 1), _torsion_key(golden_records[5][1], 2), _torsion_key(golden_records[7][1], 4)]
    row = ctypes.create_string_buffer(96 * KEY_HALF)
    for pk in keys:
        A = O.point_decode(pk)
        for p in (0, 1, 15, 30, 31) + tuple(rnd.sample(range(2, 30), 2)):
            assert emu.emu_keyset_row(row, pk, p) == F_AC | F_AOK
            for j in (0, 1, 2, 63, 126, 127) + tuple(rnd.sample(range(3, 126), 3)):
                want = _affine_entry(O._mul_int((j + 1) << (KEY_BITS * p), A))
                assert row.raw[96 * j: 96 * (j + 1)] == want, (pk.hex(), p, j)
    # keys that never reach the fast path: their facts, and a comb of identities
    # (pt_is_small_order_bytes is checked against the weak-key list in test_emu_device_math.py)
    ident = _affine_entry(O.IDENTITY)
    for pk in WEAK_KEYS + [bytes([0xEF]) + b"\xff" * 31, bytes([0x20]) + b"\xff" * 30 + b"\x7f", bytes([0x20]) + b"\xff" * 30 + b"\xff"]:
        facts = (F_AC if O.point_is_canonical(pk) else 0) | (F_AS if emu.emu_point_checks(pk) & 2 else 0) | (F_AOK if coracle.point_decode_ok(pk) else 0)
        assert facts & (F_AC | F_AS | F_AOK) != F_AC | F_AOK
        assert emu.emu_keyset_row(row, pk, 31) == facts
        assert row.raw[:96] == ident and row.raw[-96:] == ident


def test_keyed_verifier_statuses(emu, coracle, golden_records):
    """The keyed verifier returns the reference's EdDSA and Schnorr status for every mutation class of
    helpers.mutate_signature (the mutated key is the registered key) and for both halves of make_mixed_order_sigs."""
    seen = set()
    for kind in range(24):
        for r in (1, 40, 77):
            rec, other = golden_records[r + kind], golden_records[r + kind + 7]
            pk, msg, sig = mutate_signature(kind, rec, other)
            for sch in (0, 1):
                want = coracle.schnorr_verify(pk, msg, sig) if sch else coracle.eddsa_verify(pk, msg, sig)
                assert emu.emu_keyset_verify(sch, pk, msg, len(msg), sig) == want, (kind, r, sch)
                seen.add(want)
    assert seen == {0, 2, 3, 4, 5, 6, 7, 8}
    good, bad = make_mixed_order_sigs(12, seed=3)
    for sch in (0, 1):
        for pk, msg, sig in good:
            assert emu.emu_keyset_verify(sch, pk, msg, len(msg), sig) == 0
        for pk, msg, sig in bad:
            assert coracle.schnorr_verify(pk, msg, sig) == 8
            assert emu.emu_keyset_verify(sch, pk, msg, len(msg), sig) == 8


def test_keyed_verifier_message_lengths(emu, coracle, golden_records):
    """Empty messages and messages of several SHA-512 blocks under one registered key."""
    seed, pk, _, _ = golden_records[2]
    assert O.eddsa_public(seed) == pk
    rnd = random.Random(5)
    for mlen in (0, 1, 63, 64, 111, 112, 128, 300):
        msg = rnd.randbytes(mlen)
        sig = O.eddsa_sign(seed, msg)
        for sch in (0, 1):
            assert emu.emu_keyset_verify(sch, pk, msg, mlen, sig) == 0
            bent = bytearray(sig)
            bent[40] ^= 4
            want = coracle.schnorr_verify(pk, msg, bytes(bent)) if sch else coracle.eddsa_verify(pk, msg, bytes(bent))
            assert emu.emu_keyset_verify(sch, pk, msg, mlen, bytes(bent)) == want
