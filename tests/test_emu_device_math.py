"""Host emulation of the per-thread device math (tests/emu/emu.cpp compiles the SAME headers the
GPU kernels inline, with KB_HOST_EMU) against the oracles.  CPU only.  This is how the field /
curve / scalar / hash / verify / Pippenger logic is checked on a machine with no GPU; the PTX
carry-chain primitives themselves are tested on the device, at their carry and wrap edges and bit
for bit against this host build, by tests/test_gpu_field_edges.py."""
import ctypes
import hashlib
import os
import random
import subprocess

import numpy as np
import pytest

from helpers import FE_EDGE, ROOT, half_step_special_inputs, load_c_oracle, load_sign_input, make_mixed_order_sigs, make_sig_batch
from oracle import ed25519_bigint as O

P = O.P


@pytest.fixture(scope="module")
def emu():
    d = os.path.join(ROOT, "tests", "emu")
    so = os.path.join(d, "_emu.so")
    srcs = [os.path.join(d, "emu.cpp")] + [os.path.join(ROOT, "kyber-rs_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "kyber-rs_b200", "csrc")) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unused-function", "-o", so, os.path.join(d, "emu.cpp")])
    E = ctypes.CDLL(so)
    E.emu_sha512_ram.argtypes = [ctypes.c_char_p] * 4 + [ctypes.c_uint64]
    E.emu_sig_verify.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint64, ctypes.c_char_p]
    E.emu_joint4.argtypes = [ctypes.c_char_p] * 6
    E.emu_sig_verify_half.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_int]
    E.emu_sc_half.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
    E.emu_eddsa_sign.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint64]
    E.emu_msm.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    E.emu_pubpoly_eval.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_uint32]
    E.emu_dkg_fd.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    E.emu_fd_power_table.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    return E


def b32(x):
    return x.to_bytes(32, "little")


def test_field_ops(emu):
    def feop(op, a, b=bytes(32)):
        out = ctypes.create_string_buffer(32)
        emu.emu_fe_op(op, out, a, b)
        return out.raw

    rnd = random.Random(7)
    edge = list(FE_EDGE)
    vals = edge + [rnd.getrandbits(256) for _ in range(150)]
    for x in vals:
        for y in rnd.sample(vals, 8) + edge[:8]:
            assert feop(0, b32(x), b32(y)) == b32(x * y % P)
            assert feop(2, b32(x), b32(y)) == b32((x + y) % P)
            assert feop(3, b32(x), b32(y)) == b32((x - y) % P)
        assert feop(1, b32(x)) == b32(x * x % P)
        assert feop(6, b32(x)) == b32(x % P)
        # every selectable body (fe.cuh: natural and zero-free row order, borrow-mask wrap)
        assert feop(10, b32(x)) == feop(11, b32(x)) == b32(x * x % P)
        for y in edge + rnd.sample(vals, 4):
            assert feop(8, b32(x), b32(y)) == feop(9, b32(x), b32(y)) == b32(x * y % P)
            assert feop(12, b32(x), b32(y)) == b32((x - y) % P)
    # both reductions of a 512-bit value (hi : lo): the multiplications by 38 and the shift form (-DKB_FE_FOLD_SHIFT)
    for lo in vals[:60]:
        for hi in edge + rnd.sample(vals, 4):
            assert feop(13, b32(lo), b32(hi)) == feop(14, b32(lo), b32(hi)) == b32((lo + (hi << 256)) % P)
    # both multiplication bodies (schoolbook and one level of Karatsuba), incl. operands whose halves are equal,
    # ordered either way, all ones / all zeros — the sign and borrow paths of the Karatsuba differences
    M128 = 2**128
    halves = [0, 1, M128 - 1, 2**127, 0x0123456789abcdef0123456789abcdef, 2**32 - 1, 2**96]
    structured = [lo + M128 * hi for lo in halves for hi in halves]
    for x in structured:
        for y in rnd.sample(structured, 6) + rnd.sample(vals, 3):
            want = b32(x * y % P)
            assert feop(7, b32(x), b32(y)) == want, (hex(x), hex(y))
            assert feop(8, b32(x), b32(y)) == want
    for x in vals:
        for y in rnd.sample(vals, 4):
            assert feop(7, b32(x), b32(y)) == b32(x * y % P)
    for x in vals[:40]:
        assert feop(4, b32(x)) == b32(pow(x, P - 2, P))
        assert feop(5, b32(x)) == b32(pow(x, (P - 5) // 8, P))


def test_points_and_checks(emu, coracle, golden_records):
    def recode(s):
        out = ctypes.create_string_buffer(32)
        return out.raw if emu.emu_point_recode(out, s) else None

    for _, pk, sig, _ in golden_records[:64]:
        assert recode(pk) == pk and recode(sig[:32]) == sig[:32]
    rnd = random.Random(3)
    for _ in range(200):
        s = rnd.randbytes(32)
        assert recode(s) == coracle.point_recode(s)
    for k in O.WEAK_KEYS:
        assert recode(k) == coracle.point_recode(k)
        assert emu.emu_point_checks(k) & 2
    for b0 in range(256):
        for top in (0x7F, 0xFF, 0x7E):
            e = bytes([b0]) + b"\xff" * 30 + bytes([top])
            assert (emu.emu_point_checks(e) & 1) == O.point_is_canonical(e)


def test_scalars_and_hash(emu):
    rnd = random.Random(5)
    out = ctypes.create_string_buffer(32)
    for _ in range(200):
        d = rnd.randbytes(64)
        emu.emu_sc_reduce512(out, d)
        assert out.raw == O.scalar_set_bytes(d)
        a, b, c = rnd.randbytes(32), rnd.randbytes(32), rnd.randbytes(32)
        emu.emu_sc_muladd(out, a, b, c)
        assert out.raw == O.sc_mul_add(a, b, c)
    for a in (rnd.randbytes(32), b32(1), b32(O.L - 1), bytes(32), b"\xff" * 32):
        emu.emu_sc_invert(out, a)
        assert out.raw == O.sc_inv(a)
    for d in (b"\xff" * 64, bytes(64)):
        emu.emu_sc_reduce512(out, d)
        assert out.raw == O.scalar_set_bytes(d)
    for k in range(-3, 3):
        assert bool(emu.emu_sc_is_canonical(b32(O.L + k))) == (k < 0)
    dg = ctypes.create_string_buffer(64)
    for n in (0, 1, 3, 47, 48, 55, 56, 63, 64, 65, 100, 128, 191, 192, 193, 500):
        r, a, m = rnd.randbytes(32), rnd.randbytes(32), rnd.randbytes(n)
        emu.emu_sha512_ram(dg, r, a, m, n)
        assert dg.raw == hashlib.sha512(r + a + m).digest()


def test_scalar_mults(emu, coracle, golden_records):
    rnd = random.Random(11)
    out = ctypes.create_string_buffer(32)
    for _, pk, _, _ in golden_records[:24]:
        for ct in (0, 1):
            for s in (rnd.randbytes(32), rnd.randbytes(31) + b"\x0f", b"\xff" * 32, bytes(32)):
                emu.emu_mul(out, s, pk, ct)
                assert out.raw == coracle.mul(s, pk)
                emu.emu_mul_base(out, s, ct)
                assert out.raw == coracle.mul_base(s)
    # public scalars through the shared comb, including every out-of-domain shape of the top digit (SURVEY §A3)
    edge = [bytes(32), b"\xff" * 32, b32(O.L), b32(O.L - 1), b32(2**252), b32(2**253 - 1), b32(2**255 - 1), b32(2**255), b"\x88" * 31 + b"\x08", b"\x88" * 32, b"\x77" * 31 + b"\xf7"]
    for s in edge + [rnd.randbytes(32) for _ in range(300)] + [rnd.randbytes(31) + bytes([t]) for t in range(0, 256, 5)]:
        emu.emu_mul_base_comb(out, s)
        assert out.raw == coracle.mul_base(s), s.hex()


def test_verify_state_machine(emu, coracle, golden_records):
    """Every mutation class, both verifiers, against the C oracle (itself pinned to the big-int
    oracle and the reference's vectors in test_oracle_golden.py)."""
    pks, msgs, sigs = make_sig_batch(golden_records[:256:3], 24 * 6, bad_every=1)
    seen = set()
    for pk, msg, sig in zip(pks, msgs, sigs):
        for sch in (0, 1):
            want = coracle.schnorr_verify(pk, msg, sig) if sch else coracle.eddsa_verify(pk, msg, sig)
            assert emu.emu_sig_verify(sch, pk, msg, len(msg), sig) == want
            seen.add(want)
    assert seen == {0, 2, 3, 4, 5, 6, 7, 8}
    for _, pk, sig, msg in golden_records[::32]:
        assert emu.emu_sig_verify(0, pk, msg, len(msg), sig) == 0
        assert emu.emu_sig_verify(1, pk, msg, len(msg), sig) == 0


def test_half_size_lattice_step(emu):
    """sc_half (csrc/half.cuh): u odd and positive, v == u*h (mod 8L), bits = max bit length; about 128 bits
    for hash-like h, and still a valid (if long) vector for adversarial h."""
    rnd = random.Random(23)
    out = ctypes.create_string_buffer(64)
    N = 8 * O.L
    special = half_step_special_inputs()
    worst = 0
    for k in range(len(special) + 20000):
        h = special[k] if k < len(special) else rnd.randrange(O.L)
        r = emu.emu_sc_half(out, b32(h))
        bits, vneg = r & 0xFFFF, r >> 16
        u = int.from_bytes(out.raw[:32], "little")
        v = int.from_bytes(out.raw[32:], "little")
        assert u & 1 and u > 0
        assert (u * h - (-v if vneg else v)) % N == 0
        assert bits == max(u.bit_length(), v.bit_length(), 1) and bits <= 253
        if k >= len(special):
            worst = max(worst, bits)
    assert worst <= 140   # 33 or 34 radix-16 windows for honest challenges


def test_joint_radix4_digits_and_table(emu, golden_records):
    """The joint loop of the half-size-scalar verifier: the digit pairs read from x + 0x55..55 are signed radix-4 digits
    in [-1, 2] of u and v (sign of the pair pulled out, one code per pair), and the 11 table entries are i*R + j*A."""
    import random
    rng = random.Random(7)
    # code -> (du, dv): code = du * 5 + dv with du in {0, 1, 2}, dv in {-2 .. 2}
    pairs = {du * 5 + dv: (du, dv) for du in range(3) for dv in range(-2, 3)}
    pk, rb = golden_records[3][1], golden_records[4][2][:32]
    A, R = O.point_decode(pk), O.point_decode(rb)
    codes = ctypes.create_string_buffer(128)
    table = ctypes.create_string_buffer(12 * 32)
    for bits in (1, 2, 64, 127, 128, 129, 200, 253):
        for _ in range(4):
            u, v = rng.getrandbits(bits) | (1 << (bits - 1)), rng.getrandbits(bits)
            emu.emu_joint4(codes, table, u.to_bytes(32, "little"), v.to_bytes(32, "little"), pk, rb)
            su = sv = 0
            for i, c in enumerate(codes.raw):
                c = c - 256 if c > 127 else c
                du, dv = pairs[abs(c)]
                assert (du, dv) != (2, -2) and -1 <= du <= 2 and -2 <= dv <= 2
                sgn = -1 if c < 0 else 1
                assert -1 <= sgn * du <= 2 and -1 <= sgn * dv <= 2
                su += sgn * du * 4**i
                sv += sgn * dv * 4**i
            assert (su, sv) == (u, v)
            top = max(u.bit_length(), v.bit_length()) // 2 + 1   # sc_joint4_pairs: no digit at or above it
            assert not any(codes.raw[top:])
    want = {1: (0, 1), 2: (0, 2), 3: (1, -2), 4: (1, -1), 5: (1, 0), 6: (1, 1), 7: (1, 2), 9: (2, -1), 10: (2, 0), 11: (2, 1), 12: (2, 2)}
    for code, (i, j) in want.items():
        Q = O.point_add(O._mul_int(i, R), O._mul_int(j % (8 * O.L), A))
        assert table.raw[32 * (code - 1): 32 * code] == O.point_encode(Q), code


def test_verify_half_state_machine(emu, coracle, golden_records):
    """The half-size-scalar verifier returns the reference's status for every mutation class, for valid and
    near-miss signatures under keys with a small-order component, and independently of how many windows the
    block-uniform loop is forced to run."""
    pks, msgs, sigs = make_sig_batch(golden_records[1:256:3], 24 * 4, bad_every=1)
    seen = set()
    for pk, msg, sig in zip(pks, msgs, sigs):
        for sch in (0, 1):
            want = coracle.schnorr_verify(pk, msg, sig) if sch else coracle.eddsa_verify(pk, msg, sig)
            assert emu.emu_sig_verify_half(sch, pk, msg, len(msg), sig, 0) == want
            seen.add(want)
    assert seen == {0, 2, 3, 4, 5, 6, 7, 8}
    for k, (_, pk, sig, msg) in enumerate(golden_records[::16]):
        for sch in (0, 1):
            assert emu.emu_sig_verify_half(sch, pk, msg, len(msg), sig, (0, 34, 40, 64)[k % 4]) == 0
    good, bad = make_mixed_order_sigs(12)
    for sch in (0, 1):
        for pk, msg, sig in good:
            assert O.eddsa_verify(pk, msg, sig) == 0 and coracle.eddsa_verify(pk, msg, sig) == 0
            assert emu.emu_sig_verify_half(sch, pk, msg, len(msg), sig, 0) == 0
            assert emu.emu_sig_verify(sch, pk, msg, len(msg), sig) == 0
        for pk, msg, sig in bad:
            assert O.schnorr_verify(pk, msg, sig) == 8 and coracle.schnorr_verify(pk, msg, sig) == 8
            assert emu.emu_sig_verify_half(sch, pk, msg, len(msg), sig, 0) == 8
            assert emu.emu_sig_verify(sch, pk, msg, len(msg), sig) == 8


def test_verify_oracles_agree_on_mutations(coracle, golden_records):
    pks, msgs, sigs = make_sig_batch(golden_records[:48], 48, bad_every=1)
    for pk, msg, sig in zip(pks, msgs, sigs):
        assert coracle.eddsa_verify(pk, msg, sig) == O.eddsa_verify(pk, msg, sig)
        assert coracle.schnorr_verify(pk, msg, sig) == O.schnorr_verify(pk, msg, sig)


def test_pubpoly_short_horner(emu, coracle, golden_records):
    commits = [r[1] for r in golden_records[:7]]
    t8 = O.point_encode(O.point_add(O.point_decode(commits[1]), O.point_decode(O.WEAK_KEYS[2])))
    out = ctypes.create_string_buffer(32)
    for cs in (commits, [commits[0], t8] + commits[2:]):   # second: torsion-contaminated (SURVEY §7-H2)
        flat = b"".join(cs)
        for idx in (0, 1, 2, 6, 255, 1023, 65535, 2**32 - 1):
            assert emu.emu_pubpoly_eval(out, flat, len(cs), idx) == 1
            assert out.raw == coracle.pubpoly_eval(cs, idx)


def test_dkg_forward_differences(emu, coracle, golden_records):
    """csrc/dkgfd.cuh (coefficient blocks, binomial-basis Horner conversion, difference steps with the dead orders
    dropped, Straus combination with the x^(q h) mod 8L table) on one dealer: every P(i + 1) equals PubPoly::eval, also
    for a polynomial whose commitments carry small-order components (only integer-linear identities are used), for
    n < t, n = t and n > t, for 1..4 blocks of equal and unequal length."""
    commits = [r[1] for r in golden_records[100:170]]
    t8 = O.point_decode(O.WEAK_KEYS[2])
    tors = list(commits)
    tors[1] = O.point_encode(O.point_add(O.point_decode(tors[1]), t8))
    tors[5] = O.point_encode(O.point_add(O.point_decode(tors[5]), O.point_add(t8, t8)))
    cases = ((commits, 1, 4, 1), (commits, 2, 5, 1), (commits, 2, 5, 2), (commits, 3, 3, 2), (commits, 9, 4, 1), (commits, 9, 12, 4), (commits, 12, 30, 3), (tors, 7, 20, 1), (tors, 7, 20, 3),
             (commits, 33, 40, 1), (commits, 33, 70, 2), (tors, 40, 44, 4), (tors, 41, 36, 3), (commits, 70, 75, 2), (commits, 67, 34, 4))
    for cs, t, n, parts in cases:
        flat = b"".join(cs[:t])
        out = ctypes.create_string_buffer(32 * n)
        assert emu.emu_dkg_fd(out, flat, t, n, parts) == 1
        for i in range(n):
            assert out.raw[32 * i:32 * i + 32] == coracle.pubpoly_eval(cs[:t], i), (t, n, parts, i)
    assert emu.emu_dkg_fd(ctypes.create_string_buffer(32), coracle_bad_point(coracle), 1, 1, 1) == 0


def test_fd_power_table(emu):
    """kb_fd_power_table (host integers in csrc/dkgfd.cuh): (i+1)^(q h) mod 8L in signed form, magnitude <= 4L, at
    BASELINE config 4's shape (n = 1024, t = 683 in 4 blocks of 171) and a few others."""
    N = 8 * O.L
    for n, h, parts in ((1024, 171, 4), (300, 228, 3), (64, 1, 2), (17, 256, 2)):
        buf = (ctypes.c_uint32 * (9 * n * (parts - 1)))()
        emu.emu_fd_power_table(buf, n, h, parts)
        for i in range(n):
            for q in range(1, parts):
                o = 9 * (i * (parts - 1) + (q - 1))
                mag = sum(buf[o + k] << (32 * k) for k in range(8))
                neg = buf[o + 8]
                assert neg in (0, 1) and mag <= 4 * O.L
                assert (-mag if neg else mag) % N == pow(i + 1, q * h, N), (n, h, parts, i, q)


def coracle_bad_point(coracle):
    k = 0
    while coracle.point_decode_ok(bytes([k]) + b"\x13" * 31):
        k += 1
    return bytes([k]) + b"\x13" * 31


def test_pippenger_stages(emu, coracle, golden_records):
    pks = np.frombuffer(b"".join(r[1] for r in golden_records), dtype=np.uint8).reshape(-1, 32)
    rng = np.random.default_rng(1)

    def run(s, p, c=0, k=0):
        out = ctypes.create_string_buffer(32)
        bad = emu.emu_msm(out, s.shape[0], s.ctypes.data, p.ctypes.data, c, k)
        return out.raw, bad

    for n, c in [(1, 0), (2, 4), (17, 4), (50, 5), (300, 6), (700, 0), (500, 8)]:
        s = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)   # includes out-of-domain scalars (a[31] > 127)
        p = pks[:n].copy()
        want = coracle.msm(s, p)
        for k in (0, 32, 128):   # entries per accumulation thread
            got, bad = run(s, p, c, k)
            assert bad == 0 and got == want
    n = 200
    p = pks[:n].copy()
    same = np.tile(rng.integers(0, 256, size=(1, 32), dtype=np.uint8), (n, 1))   # one giant bucket per window
    assert run(same, p, 4)[0] == coracle.msm(same, p)
    z = np.zeros((n, 32), dtype=np.uint8)
    assert run(z, p)[0] == coracle.msm(z, p)
    z[:, 0] = 1
    assert run(z, p, 5)[0] == coracle.msm(z, p)
    bad_pt = p.copy()
    bad_pt[3] = np.frombuffer(hashlib.sha256(b"x").digest(), dtype=np.uint8)
    if not coracle.point_decode_ok(bad_pt[3].tobytes()):
        assert run(z, bad_pt)[1] == 1


def test_ref10_limb_wire_format(emu, coracle):
    """serde wire format of the reference (raw 4 x 10 i32 limbs, SURVEY §8f-3): real elements produced by the
    oracle's ge_scalarmult_base (un-normalised Z) and arbitrary i32 limb values."""
    rnd = random.Random(17)
    out = ctypes.create_string_buffer(32)
    for _ in range(40):
        limbs = coracle.mul_base_limbs(rnd.randbytes(32))
        emu.emu_limbs_tobytes(out, limbs.ctypes.data_as(ctypes.c_void_p))
        assert out.raw == coracle.limbs_tobytes(limbs)
    rng = np.random.default_rng(3)
    for scale in (2**10, 2**26, 2**31 - 1):
        for _ in range(30):
            limbs = rng.integers(-scale, scale, size=40, dtype=np.int64).astype(np.int32)
            emu.emu_limbs_tobytes(out, limbs.ctypes.data_as(ctypes.c_void_p))
            # the oracle's i32 limb arithmetic is only exact for limbs inside the ref10 bounds: compare with big ints
            off = [0, 26, 51, 77, 102, 128, 153, 179, 204, 230]
            val = [sum(int(limbs[10 * c + i]) << off[i] for i in range(10)) % P for c in range(3)]
            zi = pow(val[2], P - 2, P)
            x, y = val[0] * zi % P, val[1] * zi % P
            want = bytearray(b32(y))
            want[31] ^= (x & 1) << 7
            assert out.raw == bytes(want)


def test_eddsa_sign_golden(emu, golden_records):
    """EdDSA::sign (eddsa_sig.rs:120-152) + key derivation (curve.rs:74-87) as the signing kernels compose them:
    reproduces the reference's golden signatures and public keys (tests/sign/eddsa.rs:37-94)."""
    sig = ctypes.create_string_buffer(64)
    pk = ctypes.create_string_buffer(32)
    for seed, want_pk, want_sig, msg in golden_records[::24] + golden_records[:4]:
        emu.emu_eddsa_sign(sig, pk, seed, msg, len(msg))
        assert pk.raw == want_pk and sig.raw == want_sig
