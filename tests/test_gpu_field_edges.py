"""The field, scalar and lattice arithmetic of csrc/ at its carry and wrap edges.

tests/gpu_math/math_harness.cu exposes the per-thread bodies of fe.cuh and the lattice step sc_half of half.cuh as batch
entry points, and is built three ways: `emu` (plain host C++ with KB_HOST_EMU, the twin of every PTX carry chain),
`gpu-rows` (sm_100a with the default bodies) and `gpu-rip` (sm_100a with -DKB_FE_MUL_RIP -DKB_FE_SQ_RIP -DKB_FE_SUBMASK,
the bodies the verify and key-set units ship).  Every case checks that the raw result is the big-integer result mod p
and, on the GPU builds, that its raw words equal the host build's: the bodies are bit-exact with each other, so raw
equality also confirms that the host emulation the CPU suite relies on is a faithful model of the device.

Random operands almost never reach the second wrap of fe_add / fe_sub, a carry that ripples through many all-ones
words, or the top words of the squaring merge and the Karatsuba join; the inputs here are built to reach them: values
within a few units of p, 2p and multiples of 2^256, runs of 0xffffffff words, and products of the form 2^2k - 1.

The scalar kernels (Scalar::mul_add, Scalar::inv, set_bytes on a 64-byte digest) are checked through the product's own
C ABI at the edges of L and of the three folds of sc_reduce512.  The `emu` cases run without a GPU and prove the
references and input generators; the harness is also compiled for sm_100a in the CPU suite."""
import ctypes
import functools
import importlib
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

from helpers import FE_EDGE, L_ORDER, P_FIELD, ROOT, half_step_special_inputs, xof_bytes

P = P_FIELD
L = L_ORDER
M = 2**256
CSRC = os.path.join(ROOT, "kyber-rs_b200", "csrc")
HARNESS_SRC = os.path.join(ROOT, "tests", "gpu_math", "math_harness.cu")
GPU_DEFINES = {"gpu-rows": [], "gpu-rip": ["-DKB_FE_MUL_RIP", "-DKB_FE_SQ_RIP", "-DKB_FE_SUBMASK"]}
# fe_batch op numbers, in the order of the enum in math_harness.cu
OPS = {name: i for i, name in enumerate(["fe_mul", "fe_sq", "fe_add", "fe_sub", "fe_neg", "fe_mul_rows", "fe_mul_rip", "fe_mul_karatsuba", "fe_sq_rows", "fe_sq_rip",
                                         "fe_reduce512_mul", "fe_reduce512_shift", "fe_canon", "fe_is_negative", "fe_is_zero", "fe_invert", "fe_pow22523"])}
HALF_OUT_WORDS = 18

BACKENDS = [pytest.param("emu", id="emu"), pytest.param("gpu-rows", id="gpu-rows", marks=pytest.mark.gpu), pytest.param("gpu-rip", id="gpu-rip", marks=pytest.mark.gpu)]
# limb-pattern operands per backend: a fixed subset on the host build, the whole sample on the device
LIMB_SAMPLES = {"emu": 2**13, "gpu-rows": 2**20, "gpu-rip": 2**20}


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
        if nvcc is None:
            raise RuntimeError("nvcc not found: the device build of the math harness needs the CUDA toolkit")
        cmd = [nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared", "-diag-suppress", "177"] + GPU_DEFINES[backend]
    cmd += ["-I", CSRC, "-o", str(out), HARNESS_SRC]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, f"building the {backend} math harness failed:\n{' '.join(cmd)}\n{r.stdout}{r.stderr}"
    return str(out)


class Harness:
    """ctypes view of one build of math_harness.cu."""

    def __init__(self, path):
        self.lib = ctypes.CDLL(path)
        self.lib.fe_batch.argtypes = [ctypes.c_int, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        self.lib.half_batch.argtypes = [ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]

    def fe(self, op, a, b=None):
        """Raw 8-word results of `op` on the rows of a (and b): (n, 8) uint32."""
        b = np.zeros_like(a) if b is None else b
        assert a.shape == b.shape and a.dtype == b.dtype == np.uint32 and a.flags.c_contiguous and b.flags.c_contiguous
        out = np.empty_like(a)
        rc = self.lib.fe_batch(OPS[op], a.shape[0], a.ctypes.data, b.ctypes.data, out.ctypes.data)
        assert rc == 0, f"fe_batch({op}) returned {rc}"
        return out

    def half(self, h):
        out = np.empty((h.shape[0], HALF_OUT_WORDS), dtype=np.uint32)
        rc = self.lib.half_batch(h.shape[0], h.ctypes.data, out.ctypes.data)
        assert rc == 0, f"half_batch returned {rc}"
        return out


@pytest.fixture(scope="module")
def harnesses(tmp_path_factory):
    d = tmp_path_factory.mktemp("math_harness")

    @functools.cache
    def get(backend):
        return Harness(build_harness(backend, d / f"{backend}.so"))

    return get


# ---------------------------------------------------------------------------------------------------------------------
# inputs and big-integer references
# ---------------------------------------------------------------------------------------------------------------------
def words(vals):
    """ints < 2^256 -> (n, 8) little-endian uint32 words"""
    return np.frombuffer(b"".join(v.to_bytes(32, "little") for v in vals), dtype="<u4").reshape(-1, 8).astype(np.uint32)


def ints(w):
    """(n, k) uint32 words -> ints"""
    buf = np.ascontiguousarray(w, dtype="<u4").tobytes()
    k = 4 * w.shape[1]
    return [int.from_bytes(buf[i:i + k], "little") for i in range(0, len(buf), k)]


def dedup(vals):
    return list(dict.fromkeys(vals))


# FE_EDGE plus 2p - 1, 2p (2p = 2^256 - 38), 2^256 - 37, 2^256 - 2^224, and 2^32k - 1, 2^32k: a run of all-ones words, or
# a single carry target, at every word boundary
EDGE = dedup(FE_EDGE + [2 * P - 1, 2 * P, M - 37, M - 2**224] + [2**(32 * k) + d for k in range(1, 8) for d in (-1, 0)])

LIMB_WORDS = np.array([0, 1, 19, 38, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF], dtype=np.uint32)


def limb_patterns(seed, n):
    """n values whose 8 words are drawn from LIMB_WORDS: first the 8 uniform values (all-0xffffffff among them) and the
    56 single-word ones, then a deterministic sample of the 8^8."""
    head = [np.full(8, w, dtype=np.uint32) for w in LIMB_WORDS]
    for pos in range(8):
        for w in LIMB_WORDS[1:]:
            v = np.zeros(8, dtype=np.uint32)
            v[pos] = w
            head.append(v)
    idx = np.frombuffer(xof_bytes(seed, 8 * n), dtype=np.uint8) & 7
    out = LIMB_WORDS[idx].reshape(n, 8)
    out[:len(head)] = np.array(head)
    return out


def limb_pattern_pairs(seed, n):
    """(a, b): all pairs of the 64 head patterns first, then independent samples"""
    a, b = limb_patterns(seed + "/a", n), limb_patterns(seed + "/b", n)
    head = limb_patterns(seed, 64)
    a[:64 * 64] = np.repeat(head, 64, axis=0)
    b[:64 * 64] = np.tile(head, (64, 1))
    return a, b


def ripple_pairs():
    """products with long carry ripples: (2^k - 1)(2^k + 1) = 2^2k - 1, (2^k - 1)^2, and 2^j * 2^k"""
    out = []
    for k in range(32, 256):
        out += [(2**k - 1, 2**k + 1), (2**k - 1, 2**k - 1)]
    out += [(2**j, 2**k) for j in range(256) for k in range(256)]
    return out


def add_wrap_pairs(rnd):
    """a + b in [2^256 - 40, 2^256 + 40] and [2^257 - 80, 2^257 - 2] (the largest sum): the second wrap of fe_add"""
    out = []
    for s in list(range(M - 40, M + 41)) + list(range(2 * M - 80, 2 * M - 1)):
        lo, hi = max(0, s - (M - 1)), min(M - 1, s)
        out += [(a, s - a) for a in sorted({lo, hi, (lo + hi) // 2, rnd.randint(lo, hi)})]
    return out


def sub_wrap_pairs(rnd):
    """a - b in [-40, 0) and (-2^256, -2^256 + 40]: the second borrow of fe_sub"""
    out = []
    for d in list(range(-40, 0)) + list(range(-M + 1, -M + 41)):
        lo, hi = 0, M - 1 + d
        out += [(a, a - d) for a in sorted({lo, hi, (lo + hi) // 2, rnd.randint(lo, hi)})]
    return out


def karatsuba_halves():
    """operands whose 128-bit halves are equal, ordered either way, all ones or all zeros: the sign and borrow paths of
    the Karatsuba differences (the `halves` set of test_emu_device_math.py::test_field_ops)"""
    halves = [0, 1, 2**128 - 1, 2**127, 0x0123456789ABCDEF0123456789ABCDEF, 2**32 - 1, 2**96]
    vals = [lo + 2**128 * hi for lo in halves for hi in halves]
    return [(x, y) for x in vals for y in vals]


def reduction_pairs(rnd):
    """(lo, hi) with lo + 38 hi within 40 of m 2^256, m = 1..39, from both sides: every value of the word folded last and
    both of its wraps; hi takes random words, and runs of all-ones and of zero words"""
    out = []
    for m in range(1, 40):
        for d in range(-40, 41):
            t = m * M + d
            hmin, hmax = max(0, -(-(t - M + 1) // 38)), min(M - 1, t // 38)   # 0 <= lo = t - 38 hi < 2^256
            if hmin > hmax:
                continue
            his = {hmin, hmax, rnd.randint(hmin, hmax)}
            for k in (2, 5, 7):
                mask = 2**(32 * k) - 1
                for fill in (0, mask):
                    h = (rnd.randint(hmin, hmax) & ~mask) | fill
                    if hmin <= h <= hmax:
                        his.add(h)
            out += [(t - 38 * h, h) for h in sorted(his)]
    return out


def residues(vals, exact=False):
    """The raw results that are correct for the big-integer results `vals` (in [0, p)), as word arrays: an fe is any
    integer in [0, 2^256) congruent to its value (fe.cuh), so v, v + p and, for v < 38, v + 2p < 2^256; exact: v only
    (fe_canon, and the 0/1 answers of fe_is_negative / fe_is_zero)."""
    if exact:
        return (words(vals),)
    return words(vals), words([v + P for v in vals]), words([v + 2 * P if v < 38 else v for v in vals])


def canon_edges():
    """values around p, 2p and 2^256, and 0: every branch of fe_canon"""
    vals = list(range(P - 40, P + 41)) + list(range(2 * P - 40, min(2 * P + 41, M))) + list(range(M - 40, M)) + [0]
    return dedup(vals)


class Cases:
    """Inputs (words) and big-integer references, built once per module; the limb-pattern part depends on the sample
    size, so the host build's subset does not pay for the device's sample."""

    @functools.cache
    def binary(self, n):
        rnd = random.Random(101)
        pairs = [(x, y) for x in EDGE for y in EDGE] + ripple_pairs() + add_wrap_pairs(rnd) + sub_wrap_pairs(rnd) + karatsuba_halves()
        pa, pb = limb_pattern_pairs("fe-edges/binary", n)
        a = np.concatenate([words([x for x, _ in pairs]), pa])
        b = np.concatenate([words([y for _, y in pairs]), pb])
        xs, ys = ints(a), ints(b)
        prod = residues([x * y % P for x, y in zip(xs, ys)])
        want = {"fe_add": residues([(x + y) % P for x, y in zip(xs, ys)]), "fe_sub": residues([(x - y) % P for x, y in zip(xs, ys)])}
        for op in ("fe_mul", "fe_mul_rows", "fe_mul_rip", "fe_mul_karatsuba"):
            want[op] = prod
        return a, b, want

    @functools.cache
    def unary(self, n):
        vals = dedup(EDGE + [2**k + d for k in range(256) for d in (-1, 0, 1)] + canon_edges())
        a = np.concatenate([words(vals), limb_patterns("fe-edges/unary", n)])
        xs = ints(a)
        sq = residues([x * x % P for x in xs])
        red = [x % P for x in xs]
        want = {"fe_sq": sq, "fe_sq_rows": sq, "fe_sq_rip": sq, "fe_neg": residues([-x % P for x in xs]), "fe_canon": residues(red, exact=True),
                "fe_is_negative": residues([r & 1 for r in red], exact=True), "fe_is_zero": residues([int(r == 0) for r in red], exact=True)}
        return a, want

    @functools.cache
    def reduction(self, n):
        pairs = reduction_pairs(random.Random(202)) + [(x, y) for x in EDGE for y in EDGE]
        pa, pb = limb_pattern_pairs("fe-edges/reduction", n)
        lo = np.concatenate([words([x for x, _ in pairs]), pa])
        hi = np.concatenate([words([y for _, y in pairs]), pb])
        want = residues([(x + (y << 256)) % P for x, y in zip(ints(lo), ints(hi))])
        return lo, hi, want

    @functools.cache
    def exponentiation(self):
        rnd = random.Random(303)
        vals = EDGE + [rnd.getrandbits(256) for _ in range(4096)]
        return words(vals), {"fe_invert": residues([pow(x, P - 2, P) for x in vals]), "fe_pow22523": residues([pow(x, (P - 5) // 8, P) for x in vals])}

    @functools.cache
    def half(self):
        rnd = random.Random(404)
        special = half_step_special_inputs()
        return special, special + [rnd.randrange(L) for _ in range(2**16)]


@pytest.fixture(scope="module")
def cases():
    return Cases()


# ---------------------------------------------------------------------------------------------------------------------
# checks
# ---------------------------------------------------------------------------------------------------------------------
def _item(inputs, i):
    return ", ".join(hex(int.from_bytes(np.ascontiguousarray(x[i]).astype("<u4").tobytes(), "little")) for x in inputs)


def check_fe(harnesses, backend, op, inputs, want):
    """(a) the raw result is one of the representatives `want` (see residues); (b) on the device builds, its words are
    the host build's.  A failure names the first item that differs."""
    raw = harnesses(backend).fe(op, *inputs)
    ok = np.zeros(raw.shape[0], dtype=bool)
    for w in want:
        ok |= (raw == w).all(axis=1)
    if not ok.all():
        i = int(np.nonzero(~ok)[0][0])
        pytest.fail(f"{backend} {op}: {int((~ok).sum())} of {ok.size} items wrong, first {i}: inputs ({_item(inputs, i)}): raw {_item((raw,), i)}, "
                    f"want {_item((want[0],), i)}{' (mod p)' if len(want) > 1 else ''}")
    if backend != "emu":
        host = harnesses("emu").fe(op, *inputs)
        bad = np.nonzero((raw != host).any(axis=1))[0]
        if bad.size:
            i = int(bad[0])
            pytest.fail(f"{backend} {op}: {bad.size} items differ from the host build, first {i}: inputs ({_item(inputs, i)}): raw {_item((raw,), i)}, host {_item((host,), i)}")


@pytest.mark.parametrize("backend", BACKENDS)
def test_fe_binary_ops(harnesses, cases, backend):
    """every multiplication body, fe_add and fe_sub on edge x edge, long carry ripples, the second wrap and borrow,
    Karatsuba halves and limb patterns"""
    a, b, want = cases.binary(LIMB_SAMPLES[backend])
    for op in ("fe_mul", "fe_mul_rows", "fe_mul_rip", "fe_mul_karatsuba", "fe_add", "fe_sub"):
        check_fe(harnesses, backend, op, (a, b), want[op])


@pytest.mark.parametrize("backend", BACKENDS)
def test_fe_unary_ops(harnesses, cases, backend):
    """both squaring bodies, fe_neg, and fe_canon / fe_is_negative / fe_is_zero around p, 2p and 2^256"""
    a, want = cases.unary(LIMB_SAMPLES[backend])
    for op in ("fe_sq", "fe_sq_rows", "fe_sq_rip", "fe_neg"):
        check_fe(harnesses, backend, op, (a,), want[op])
    for op in ("fe_canon", "fe_is_negative", "fe_is_zero"):   # exact results: fully reduced, 0 / 1
        check_fe(harnesses, backend, op, (a,), want[op])


@pytest.mark.parametrize("backend", BACKENDS)
def test_fe_reductions(harnesses, cases, backend):
    """both reductions of a 512-bit value (hi : lo) with lo + 38 hi near every multiple of 2^256 they can meet"""
    lo, hi, want = cases.reduction(LIMB_SAMPLES[backend])
    for op in ("fe_reduce512_mul", "fe_reduce512_shift"):
        check_fe(harnesses, backend, op, (lo, hi), want)


@pytest.mark.parametrize("backend", BACKENDS)
def test_fe_exponentiations(harnesses, cases, backend):
    """fe_invert = x^(p-2) and fe_pow22523 = x^((p-5)/8) on the edge values (0, p and 2p give 0) and random values"""
    a, want = cases.exponentiation()
    zero = [EDGE.index(v) for v in (0, P, 2 * P)]
    for op in ("fe_invert", "fe_pow22523"):
        assert not want[op][0][zero].any()
        check_fe(harnesses, backend, op, (a,), want[op])


@pytest.mark.parametrize("backend", BACKENDS)
def test_sc_half(harnesses, cases, backend):
    """sc_half (csrc/half.cuh): u odd and positive, u h = +-|v| (mod 8L), bits = max bit length <= 253, at most 140 bits
    for random challenges; bit for bit the host build's result"""
    special, hs = cases.half()
    hw = words(hs)
    out = harnesses(backend).half(hw)
    N = 8 * L
    worst = 0
    for k, (h, u, v) in enumerate(zip(hs, ints(out[:, :8]), ints(out[:, 8:16]))):
        vneg, bits = int(out[k, 16]), int(out[k, 17])
        item = f"{backend} sc_half item {k}: h = {hex(h)}: u = {hex(u)}, |v| = {hex(v)}, vneg = {vneg}, bits = {bits}"
        assert u & 1 and u > 0, item
        assert vneg in (0, 1) and (u * h - (-v if vneg else v)) % N == 0, item
        assert bits == max(u.bit_length(), v.bit_length(), 1) and bits <= 253, item
        if k >= len(special):
            worst = max(worst, bits)
    assert worst <= 140
    if backend != "emu":
        host = harnesses("emu").half(hw)
        bad = np.nonzero((out != host).any(axis=1))[0]
        assert bad.size == 0, f"{backend} sc_half: {bad.size} items differ from the host build, first {int(bad[0])}: h = {hex(hs[int(bad[0])])}"


@pytest.mark.parametrize("backend", sorted(GPU_DEFINES))
def test_math_harness_compiles_for_sm100a(tmp_path, backend):
    """The device builds of the harness compile for sm_100a without a GPU, so a broken harness fails here and not only
    on a B200."""
    if find_nvcc() is None:
        pytest.skip("nvcc not found")
    build_harness(backend, tmp_path / f"{backend}.so")


# ---------------------------------------------------------------------------------------------------------------------
# scalars mod L through the product's kernels (Context.sc_*), at the edges of L and of the folds of sc_reduce512
# ---------------------------------------------------------------------------------------------------------------------
SC_EDGE = [0, 1, 2, L - 2, L - 1, L, L + 1, 2 * L - 1, 2 * L, 2**252 - 1, 2**252, 2**253 - 1, 2**255 - 1, 2**255, M - L, M - 1]


def sc_bytes(vals, width=32):
    return np.frombuffer(b"".join(v.to_bytes(width, "little") for v in vals), dtype=np.uint8).reshape(-1, width).copy()


def check_scalars(what, got, want, inputs):
    got = [int.from_bytes(r.tobytes(), "little") for r in got]
    if got != want:
        i = next(k for k, (g, w) in enumerate(zip(got, want)) if g != w)
        pytest.fail(f"{what} item {i} of {len(want)}: inputs ({', '.join(hex(x[i]) for x in inputs)}): got {hex(got[i])}, want {hex(want[i])}")


@pytest.fixture(scope="module")
def ctx():
    kb = importlib.import_module("kyber-rs_b200")
    c = kb.Context(0)
    yield c
    c.close()


@pytest.mark.gpu
def test_sc_muladd_edges(ctx):
    """(a b + c) mod L on raw 256-bit operands: every triple of the edge set, and random triples"""
    rnd = random.Random(505)
    trip = [(a, b, c) for a in SC_EDGE for b in SC_EDGE for c in SC_EDGE]
    trip += [(rnd.getrandbits(256), rnd.getrandbits(256), rnd.getrandbits(256)) for _ in range(2**16)]
    a, b, c = ([t[k] for t in trip] for k in range(3))
    got = ctx.sc_muladd_batch(sc_bytes(a), sc_bytes(b), sc_bytes(c))
    check_scalars("sc_muladd", got, [(x * y + z) % L for x, y, z in trip], (a, b, c))


@pytest.mark.gpu
def test_sc_invert(ctx):
    """Scalar::inv = a^(L-2) mod L on raw 256-bit values (0 and L give 0, L + 1 gives 1), and a inv(a) = 1 (mod L)"""
    rnd = random.Random(606)
    vals = SC_EDGE + [rnd.getrandbits(256) for _ in range(4096)]
    inv = ctx.sc_invert_batch(sc_bytes(vals))
    want = [pow(v % L, L - 2, L) for v in vals]
    assert want[SC_EDGE.index(0)] == want[SC_EDGE.index(L)] == 0 and want[SC_EDGE.index(L + 1)] == 1
    check_scalars("sc_invert", inv, want, (vals,))
    unit = [k for k, v in enumerate(vals) if v % L]
    one = ctx.sc_muladd_batch(sc_bytes([vals[k] for k in unit]), inv[unit], np.zeros((len(unit), 32), dtype=np.uint8))
    check_scalars("a * sc_invert(a)", one, [1] * len(unit), ([vals[k] for k in unit],))


@pytest.mark.gpu
def test_sc_reduce64_edges(ctx):
    """a 64-byte digest mod L at k L + {-1, 0, 1} for k up to the largest that fits, at 2^j - 1 and 2^j for j = 252..512
    (every fold of sc_reduce512 at its top), at 2^512 - 1, and on random digests"""
    rnd = random.Random(707)
    kmax = (2**512 - 1) // L
    ks = [1, 2] + [2**i for i in range(2, kmax.bit_length())] + [kmax]
    vals = [k * L + d for k in ks for d in (-1, 0, 1)] + [2**j + d for j in range(252, 513) for d in (-1, 0)] + [2**512 - 1]
    vals = dedup(v for v in vals if 0 <= v < 2**512) + [rnd.getrandbits(512) for _ in range(2**16)]
    got = ctx.sc_reduce64_batch(sc_bytes(vals, 64))
    check_scalars("sc_reduce64", got, [v % L for v in vals], (vals,))
