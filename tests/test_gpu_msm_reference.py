"""The Pippenger MSM (csrc/msm.cuh, capi_msm.cu) against the exact closed form of tests/msm_reference.py, at every
window width, several bucket groupings, and sizes that span several 2^22-point chunks, through the host, device and
decoded-point entry points, split into partials, and across the GPUs of a box.  Needs a B200.

Sizes above 2^24 run only when KB_TEST_MSM_LOG2MAX is set (e.g. 26)."""
import importlib
import os

import numpy as np
import pytest

import msm_reference as R
from helpers import _off_curve
from oracle import ed25519_bigint as O

pytestmark = pytest.mark.gpu

CHUNK = 1 << 22
NMAX = 1 << 24
LOG2MAX = int(os.environ.get("KB_TEST_MSM_LOG2MAX", "24"))


@pytest.fixture(scope="module")
def kb():
    return importlib.import_module("kyber-rs_b200")


@pytest.fixture(scope="module")
def ctx(kb):
    c = kb.Context(0)
    yield c
    c.close()


def _ctx_env(kb, **env):
    os.environ.update(env)
    try:
        return kb.Context(0)
    finally:
        for k in env:
            del os.environ[k]


@pytest.fixture(scope="module")
def pts(ctx, coracle):
    """2^24 pairwise distinct points P_i = r_i*B + t_i*T8, generated on the GPU and sampled against the oracles."""
    return R.gpu_points(ctx, NMAX, 1, coracle)


class Refs:
    """Scalars and closed-form results, each computed once per (family, n, c) and shared by every path.  The uniform
    and reduced families are drawn once at 2^24 and sliced."""

    def __init__(self, pts):
        self.p, self.r, self.t = pts
        self.s = {}
        self.want = {}

    def scalars(self, family, n, c=16):
        if family in ("uniform", "reduced"):
            if family not in self.s:
                self.s[family] = R.FAMILIES[family](NMAX, 2, c)
            return self.s[family][:n]
        if (family, n, c) not in self.s:
            self.s[family, n, c] = R.FAMILIES[family](n, 2, c)
        return self.s[family, n, c]

    def expected(self, family, n, c=16):
        key = (family, n, 0 if family in ("uniform", "reduced") else c)
        if key not in self.want:
            self.want[key] = R.expected(self.scalars(family, n, c), self.r[:n], self.t[:n])
        return self.want[key]


@pytest.fixture(scope="module")
def refs(pts):
    return Refs(pts)


def _window_bits(n):
    return min(16, max(4, n.bit_length() - 1 - 3))


@pytest.mark.parametrize("c", range(4, 17))
def test_window_width(kb, refs, c):
    """KB_MSM_C = 4..16 at 3 * 2^12 points: raw uniform scalars, a signed-digit carry through every window, and the
    edge scalars of the effective-scalar rule."""
    n = 3 << 12
    cx = _ctx_env(kb, KB_MSM_C=str(c))
    try:
        for family in ("uniform", "carry", "edges"):
            enc, bad = cx.msm(refs.scalars(family, n, c), refs.p[:n])
            assert bad == 0 and enc == refs.expected(family, n, c), (family, c)
    finally:
        cx.close()


@pytest.mark.parametrize("n", [(1 << 15) + 1, 1 << 17, (1 << 18) + 5, 1 << 19, 1 << 20])
def test_size_rule(ctx, refs, n):
    """The window width the size rule picks (c = 12, 14, 15, 16, 16) with every scalar family."""
    c = _window_bits(n)
    for family in sorted(R.FAMILIES):
        enc, bad = ctx.msm(refs.scalars(family, n, c), refs.p[:n])
        assert bad == 0 and enc == refs.expected(family, n, c), (family, n, c)


@pytest.mark.parametrize("groups", [32, 33, 3000, 16384])
def test_bucket_groups(kb, refs, groups):
    """KB_MSM_GROUPS at 2^20 points (c = 16, 32768 buckets per window): many groups per fold thread, group counts
    that do not divide the window, and 16384 groups of two buckets."""
    n = 1 << 20
    cx = _ctx_env(kb, KB_MSM_GROUPS=str(groups))
    try:
        for family in ("uniform", "reduced", "carry"):
            enc, bad = cx.msm(refs.scalars(family, n, 16), refs.p[:n])
            assert bad == 0 and enc == refs.expected(family, n, 16), (family, groups)
    finally:
        cx.close()


@pytest.fixture(scope="module")
def dev(ctx, pts):
    """The 2^24 points on the device as encodings and as decoded (X, Y, Z, T) words, a sample of the latter scaled
    by a random lambda so that Z != 1 — across every chunk boundary among them."""
    import torch

    d = torch.device("cuda", 0)
    enc = torch.from_numpy(pts[0]).to(d)
    raw = torch.empty((NMAX, 128), dtype=torch.uint8, device=d)
    st = torch.empty(NMAX, dtype=torch.uint8, device=d)
    ctx.dev_point_decompress(NMAX, enc, raw, st)
    torch.cuda.synchronize()
    assert not st.any().item()
    rng = np.random.default_rng(17)
    idx = np.unique(np.concatenate([rng.choice(NMAX, 4096, replace=False), [0, 1, CHUNK - 1, CHUNK, CHUNK + 1, 2 * CHUNK - 1, 2 * CHUNK, 3 * CHUNK, NMAX - 1]]))
    ti = torch.from_numpy(idx).to(d)
    words = raw[ti].cpu().numpy().view("<u4").reshape(-1, 4, 8)
    for row in words:
        lam = int(rng.integers(2, 2**62)) * int(rng.integers(2, 2**62)) % O.P
        for k in range(4):
            v = sum(int(row[k, j]) << (32 * j) for j in range(8)) * lam % O.P
            row[k] = [(v >> (32 * j)) & 0xFFFFFFFF for j in range(8)]
    raw[ti] = torch.from_numpy(words.reshape(-1, 32).view(np.uint8).copy()).to(d)
    return enc, raw


def _dev_scalars(refs, family, n):
    import torch

    return torch.from_numpy(np.ascontiguousarray(refs.scalars(family, n))).to("cuda:0")


def _dev_msm(ctx, n, d_s, d_p, ext=False):
    import torch

    out = torch.zeros(32, dtype=torch.uint8, device="cuda:0")
    bad = torch.full((1,), -1, dtype=torch.int64, device="cuda:0")
    (ctx.dev_msm_ext if ext else ctx.dev_msm)(n, d_s, d_p, out, None, bad)
    torch.cuda.synchronize()
    return out.cpu().numpy().tobytes(), int(bad.item())


CHUNKED = [CHUNK, CHUNK + 1, 2 * CHUNK + (1 << 19) + 3, NMAX]


@pytest.mark.parametrize("n", CHUNKED)
def test_chunks_host_device_decoded(ctx, refs, dev, n):
    """One to four 2^22-point chunks (a one-point ragged last chunk among them) through kb_msm, kb_dev_msm and
    kb_dev_msm_ext: the partial sums are chained across chunks, and every chunk reads its own scalars and points."""
    enc, raw = dev
    families = ("uniform", "reduced") if n in (CHUNK + 1, NMAX) else ("uniform",)
    for family in families:
        want = refs.expected(family, n)
        got, bad = ctx.msm(refs.scalars(family, n), refs.p[:n])
        assert bad == 0 and got == want, ("host", family, n)
        d_s = _dev_scalars(refs, family, n)
        assert _dev_msm(ctx, n, d_s, enc[:n]) == (want, 0), ("device", family, n)
        assert _dev_msm(ctx, n, d_s, raw[:n], ext=True) == (want, 0), ("decoded", family, n)


def test_partials_split_off_chunk_boundaries(ctx, refs, dev):
    """kb_dev_msm partials over ranges cut away from the chunk boundaries, folded by kb_dev_point_sum and by
    kb_point_sum, equal the MSM of the whole range."""
    import torch

    enc, raw = dev
    n = CHUNKED[2]
    want = refs.expected("uniform", n)
    d_s = _dev_scalars(refs, "uniform", n)
    cuts = [0, 3 * (1 << 20) + 7, 2 * CHUNK + 1, n]
    for pts_dev, fn in ((enc, ctx.dev_msm), (raw, ctx.dev_msm_ext)):
        parts = torch.zeros((len(cuts) - 1, 128), dtype=torch.uint8, device="cuda:0")
        bad = torch.zeros(1, dtype=torch.int64, device="cuda:0")
        for k, (lo, hi) in enumerate(zip(cuts, cuts[1:])):
            fn(hi - lo, d_s[lo:hi], pts_dev[lo:hi], None, parts[k], bad)
        out = torch.zeros(32, dtype=torch.uint8, device="cuda:0")
        ctx.dev_point_sum(len(cuts) - 1, parts, out)
        torch.cuda.synchronize()
        assert out.cpu().numpy().tobytes() == want
        assert ctx.point_sum(parts.cpu().numpy()) == want


def test_bad_points_counted_in_every_chunk(ctx, refs, dev):
    """Undecodable encodings in chunk 0, chunk 1 and the ragged last chunk are all counted (the sum is undefined
    then); for decoded points, Z = 0 and off-curve entries in different chunks likewise."""
    import torch

    enc, raw = dev
    n = CHUNKED[2]
    where = [5, CHUNK + 7, n - 2]
    s = refs.scalars("uniform", n)
    p = refs.p[:n].copy()
    for k, i in enumerate(where):
        p[i] = np.frombuffer(_off_curve(10 + k), dtype=np.uint8)
    assert ctx.msm(s, p)[1] == 3
    d_s = _dev_scalars(refs, "uniform", n)
    assert _dev_msm(ctx, n, d_s, torch.from_numpy(p).to("cuda:0"))[1] == 3
    r2 = raw[:n].clone()
    r2[where[0], 64:96] = 0                  # Z = 0
    r2[where[1], 0] ^= 1                     # X off the curve
    r2[where[2], 32] ^= 4                    # Y off the curve
    assert _dev_msm(ctx, n, d_s, r2, ext=True)[1] == 3


def test_multi_device(kb, refs):
    """kb_mctx_msm over every visible GPU, with a point count the device count does not divide."""
    import torch

    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("a single GPU is visible")
    n = NMAX - 3
    m = kb.MultiContext(list(range(min(ngpu, 8))))
    try:
        assert m.msm(refs.scalars("uniform", n), refs.p[:n]) == (refs.expected("uniform", n), 0)
    finally:
        m.close()


@pytest.mark.skipif(LOG2MAX < 26, reason="set KB_TEST_MSM_LOG2MAX=26 to run 2^26 points")
def test_opt_in_2p26(ctx, coracle):
    """2^26 points (16 chunks) through kb_msm and kb_dev_msm."""
    import torch

    n = 1 << 26
    p, r, t = R.gpu_points(ctx, n, 3, coracle, sample=256)
    s = R.uniform(n, 3)
    want = R.expected(s, r, t)
    assert ctx.msm(s, p) == (want, 0)
    assert _dev_msm(ctx, n, torch.from_numpy(s).to("cuda:0"), torch.from_numpy(p).to("cuda:0")) == (want, 0)


def test_edge_scalars_scalar_mult(kb, ctx, coracle, refs):
    """The effective-scalar edges through fixed-base and variable-base multiplication, constant time and variable
    time, on points with torsion components and on one shared point."""
    s = R.EDGES
    m = s.shape[0]
    p = refs.p[:m].copy()
    want_b = coracle.mul_base_batch(s)
    want_p = coracle.mul_batch(s, p)
    want_1 = coracle.mul_batch(s, np.repeat(p[:1], m, axis=0))
    for flags in (0, kb.binding.FLAG_VARTIME):
        assert (ctx.point_mul_base_batch(s, flags) == want_b).all(), flags
        out, st = ctx.point_mul_batch(s, p, flags)
        assert not st.any() and (out == want_p).all(), flags
        out, st = ctx.point_mul_batch(s, p[:1], flags)
        assert not st.any() and (out == want_1).all(), flags
