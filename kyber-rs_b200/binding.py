"""ctypes binding of include/kyber_b200.h.  Pure plumbing: numpy (host) or torch (device)
buffers in, kernel launches inside the library, buffers out."""
from __future__ import annotations

import ctypes
import os

import numpy as np

LIB_PATH = os.environ.get("KYBER_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libkyber_b200.so")

FLAG_VARTIME = 1
FLAG_SHARED_POINT = 2

# kb_sig_status -> the reference's SignatureError display strings (sign/error.rs:6-25)
SIG_STATUS_NAMES = {
    0: "ok",
    1: "wrong signature length",
    2: "signature is not canonical",
    3: "R is not canonical",
    4: "R has small order",
    5: "public key is not canonical",
    6: "public key has small order",
    7: "marshalling error",
    8: "signature is not valid",
}


class KBError(RuntimeError):
    pass


_LIB = None

# every symbol include/kyber_b200.h declares (tests check the .so exports all of them)
EXPORTS = [
    "kb_ctx_create", "kb_ctx_destroy", "kb_ctx_wipe", "kb_last_error", "kb_device_sm_count", "kb_launch_count", "kb_host_alloc", "kb_host_free",
    "kb_point_mul_base_batch", "kb_point_mul_batch", "kb_point_recode_batch", "kb_point_from_limbs_batch", "kb_point_add_batch", "kb_point_check_batch", "kb_point_decompress_batch", "kb_point_compress_batch", "kb_point_eq_batch",
    "kb_sc_reduce64_batch", "kb_sc_muladd_batch", "kb_sc_invert_batch", "kb_challenge_batch", "kb_eddsa_verify_batch", "kb_schnorr_verify_batch", "kb_eddsa_sign_batch",
    "kb_pubpoly_eval_batch", "kb_vss_verify_deals_batch", "kb_dkg_verify_round", "kb_dkg_verify_round_limbs", "kb_pubpoly_sum", "kb_msm", "kb_point_sum",
    "kb_vss_session_ids", "kb_find_pub_batch", "kb_dkg_process_round", "kb_vss_rabin_verify_deals_batch", "kb_dss_verify_partials", "kb_recover_commit_batch", "kb_recover_pub_poly", "kb_dkg_resharing_key",
    "kb_dev_dkg_process_round", "kb_dev_point_decompress", "kb_dev_challenge", "kb_pripoly_eval_batch", "kb_dev_pripoly_eval",
    "kb_mctx_create", "kb_mctx_destroy", "kb_mctx_device_count", "kb_mctx_ctx", "kb_mctx_last_error", "kb_mctx_launch_count", "kb_mctx_verify_batch", "kb_mctx_point_mul_base_batch", "kb_mctx_point_mul_batch",
    "kb_mctx_dkg_verify_round", "kb_mctx_dkg_process_round", "kb_mctx_msm",
    "kb_dev_eddsa_verify", "kb_dev_point_mul_base", "kb_dev_point_mul", "kb_dev_msm", "kb_dev_msm_ext", "kb_dev_dkg_verify_round", "kb_dev_dkg_verify_round_limbs", "kb_dev_point_sum",
    "kb_probe_imad", "kb_verify_kernel_times",
    "kb_keyset_create", "kb_keyset_destroy", "kb_keyset_verify_batch", "kb_dev_keyset_verify",
    "kb_dkg_process_round_keyed", "kb_dev_dkg_process_round_keyed",
    "kb_mctx_keyset_create", "kb_mctx_keyset_destroy", "kb_mctx_keyset_verify_batch", "kb_mctx_dkg_process_round_keyed",
    "kb_keyset_mul_batch", "kb_dev_keyset_mul", "kb_mctx_keyset_mul_batch",
]


def load_library(path: str = LIB_PATH):
    """dlopen libkyber_b200.so.  Fails loudly when it has not been built (no fallback)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(path):
        raise KBError(f"{path} not found: build it with `make -C kyber-rs_b200/csrc` (or __graft_entry__.build()); there is no CPU fallback")
    L = ctypes.CDLL(path)
    vp, sz, u32, i32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_int
    L.kb_ctx_create.argtypes = [i32, ctypes.POINTER(vp)]
    L.kb_ctx_destroy.argtypes = [vp]
    L.kb_ctx_destroy.restype = None
    L.kb_ctx_wipe.argtypes = [vp]
    L.kb_last_error.argtypes = [vp]
    L.kb_last_error.restype = ctypes.c_char_p
    L.kb_device_sm_count.argtypes = [vp]
    L.kb_launch_count.argtypes = [vp]
    L.kb_launch_count.restype = ctypes.c_uint64
    L.kb_host_alloc.argtypes = [sz]
    L.kb_host_alloc.restype = vp
    L.kb_host_free.argtypes = [vp]
    L.kb_host_free.restype = None
    L.kb_point_mul_base_batch.argtypes = [vp, sz, vp, vp, u32]
    L.kb_point_mul_batch.argtypes = [vp, sz, vp, vp, vp, vp, u32]
    L.kb_point_recode_batch.argtypes = [vp, sz, vp, vp, vp]
    L.kb_point_from_limbs_batch.argtypes = [vp, sz, vp, vp]
    L.kb_point_add_batch.argtypes = [vp, sz, vp, vp, vp, vp, i32]
    L.kb_point_check_batch.argtypes = [vp, sz, vp, vp]
    L.kb_point_decompress_batch.argtypes = [vp, sz, vp, vp, vp]
    L.kb_point_compress_batch.argtypes = [vp, sz, vp, vp]
    L.kb_point_eq_batch.argtypes = [vp, sz, vp, vp, vp]
    L.kb_sc_reduce64_batch.argtypes = [vp, sz, vp, vp]
    L.kb_sc_muladd_batch.argtypes = [vp, sz, vp, vp, vp, vp]
    L.kb_sc_invert_batch.argtypes = [vp, sz, vp, vp]
    L.kb_challenge_batch.argtypes = [vp, sz, vp, vp, vp, vp, vp]
    L.kb_eddsa_verify_batch.argtypes = [vp, sz, vp, vp, vp, vp, vp]
    L.kb_schnorr_verify_batch.argtypes = [vp, sz, vp, vp, vp, vp, vp]
    L.kb_eddsa_sign_batch.argtypes = [vp, sz, vp, vp, vp, vp, vp]
    L.kb_pubpoly_eval_batch.argtypes = [vp, sz, sz, vp, sz, vp, vp, vp, vp]
    L.kb_vss_verify_deals_batch.argtypes = [vp, sz, sz, vp, sz, vp, vp, vp, vp]
    L.kb_dkg_verify_round.argtypes = [vp, sz, sz, sz, sz, vp, vp, vp]
    L.kb_dkg_verify_round_limbs.argtypes = [vp, sz, sz, sz, sz, vp, vp, vp]
    L.kb_pubpoly_sum.argtypes = [vp, sz, sz, vp, vp, vp]
    L.kb_msm.argtypes = [vp, sz, vp, vp, vp, vp, vp]
    L.kb_vss_session_ids.argtypes = [vp, sz, sz, sz, i32, vp, vp, vp, vp, vp]
    L.kb_find_pub_batch.argtypes = [vp, sz, vp, sz, vp, i32, vp]
    L.kb_dkg_process_round.argtypes = [vp, sz, sz, sz, sz, i32, vp, vp, vp] + [vp] * 10
    L.kb_dev_dkg_process_round.argtypes = [vp, sz, sz, sz, i32, vp, vp, vp] + [vp] * 10 + [vp]
    L.kb_vss_rabin_verify_deals_batch.argtypes = [vp, sz, sz, vp, vp, sz, vp, vp, vp, vp, vp]
    L.kb_dss_verify_partials.argtypes = [vp, sz, vp, vp, vp, sz, sz, vp, vp, vp, vp]
    L.kb_recover_commit_batch.argtypes = [vp, sz, sz, vp, vp, vp, vp]
    L.kb_recover_pub_poly.argtypes = [vp, sz, vp, vp, vp, vp]
    L.kb_dkg_resharing_key.argtypes = [vp, sz, sz, vp, vp, u32, vp, vp, vp, vp]
    L.kb_point_sum.argtypes = [vp, sz, vp, vp]
    L.kb_dev_eddsa_verify.argtypes = [vp, sz, vp, vp, vp, vp, vp, i32, vp]
    L.kb_dev_point_mul_base.argtypes = [vp, sz, vp, vp, u32, vp]
    L.kb_dev_point_mul.argtypes = [vp, sz, vp, vp, vp, vp, u32, vp]
    L.kb_dev_msm.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp]
    L.kb_dev_msm_ext.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp]
    L.kb_dev_dkg_verify_round.argtypes = [vp, sz, sz, sz, vp, vp, vp, vp]
    L.kb_dev_dkg_verify_round_limbs.argtypes = [vp, sz, sz, sz, vp, vp, vp, vp]
    L.kb_dev_point_sum.argtypes = [vp, sz, vp, vp, vp]
    L.kb_pripoly_eval_batch.argtypes = [vp, sz, sz, vp, sz, vp]
    L.kb_dev_pripoly_eval.argtypes = [vp, sz, sz, vp, sz, vp, vp]
    L.kb_dev_point_decompress.argtypes = [vp, sz, vp, vp, vp, vp]
    L.kb_dev_challenge.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp]
    L.kb_mctx_create.argtypes = [ctypes.POINTER(i32), i32, ctypes.POINTER(vp)]
    L.kb_mctx_destroy.argtypes = [vp]
    L.kb_mctx_destroy.restype = None
    L.kb_mctx_device_count.argtypes = [vp]
    L.kb_mctx_ctx.argtypes = [vp, i32]
    L.kb_mctx_ctx.restype = vp
    L.kb_mctx_last_error.argtypes = [vp]
    L.kb_mctx_last_error.restype = ctypes.c_char_p
    L.kb_mctx_launch_count.argtypes = [vp]
    L.kb_mctx_launch_count.restype = ctypes.c_uint64
    L.kb_mctx_verify_batch.argtypes = [vp, sz, vp, vp, vp, vp, vp, i32]
    L.kb_mctx_point_mul_base_batch.argtypes = [vp, sz, vp, vp, u32]
    L.kb_mctx_point_mul_batch.argtypes = [vp, sz, vp, vp, vp, vp, u32]
    L.kb_mctx_dkg_verify_round.argtypes = [vp, sz, sz, sz, i32, vp, vp, vp]
    L.kb_mctx_dkg_process_round.argtypes = [vp, sz, sz, sz, i32, vp, vp, vp] + [vp] * 10
    L.kb_mctx_msm.argtypes = [vp, sz, vp, vp, vp, vp]
    L.kb_probe_imad.argtypes = [vp, i32, i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    L.kb_verify_kernel_times.argtypes = [vp, i32, ctypes.POINTER(ctypes.c_float)]
    L.kb_keyset_create.argtypes = [vp, sz, vp, ctypes.POINTER(vp)]
    L.kb_keyset_destroy.argtypes = [vp]
    L.kb_keyset_destroy.restype = None
    L.kb_keyset_verify_batch.argtypes = [vp, sz, vp, vp, vp, vp, vp, i32]
    L.kb_dev_keyset_verify.argtypes = [vp, sz, vp, vp, vp, vp, vp, i32, vp]
    L.kb_keyset_mul_batch.argtypes = [vp, sz, vp, vp, vp, vp, u32]
    L.kb_dev_keyset_mul.argtypes = [vp, sz, vp, vp, vp, vp, u32, vp]
    L.kb_dkg_process_round_keyed.argtypes = [vp, vp, vp, sz, sz, sz, sz, i32, vp, vp, vp] + [vp] * 8
    L.kb_dev_dkg_process_round_keyed.argtypes = [vp, vp, vp, sz, sz, sz, sz, i32, vp, vp, vp] + [vp] * 8 + [vp]
    L.kb_mctx_keyset_create.argtypes = [vp, sz, vp, ctypes.POINTER(vp)]
    L.kb_mctx_keyset_destroy.argtypes = [vp]
    L.kb_mctx_keyset_destroy.restype = None
    L.kb_mctx_keyset_verify_batch.argtypes = [vp, sz, vp, vp, vp, vp, vp, i32]
    L.kb_mctx_keyset_mul_batch.argtypes = [vp, sz, vp, vp, vp, vp, u32]
    L.kb_mctx_dkg_process_round_keyed.argtypes = [vp, vp, vp, sz, sz, sz, i32, vp, vp, vp] + [vp] * 8
    _LIB = L
    return L


def _u8(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else None


def pack_messages(msgs):
    """list of bytes -> (flat uint8 array, uint64 offsets[n+1]) as the C ABI wants them."""
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    if len(msgs):
        off[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64)
    flat = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy() if int(off[-1]) else np.zeros(0, dtype=np.uint8)
    return flat, off


def _keyed_batches(deal, resp, m, what):
    """(ctypes args, [deal_status | None, resp_status | None], arrays to keep alive) of the two signature batches of a
    keyed round; a batch is (msg flat, msg_off[m+1], sig[m,64]) or None."""
    args, outs, keep = [], [], []
    for batch in (deal, resp):
        if batch is None:
            args += [None] * 4
            outs.append(None)
            continue
        msg, off, sig = _u8(batch[0]), np.ascontiguousarray(batch[1], dtype=np.uint64), _u8(batch[2], (-1, 64))
        if sig.shape[0] != m or off.shape[0] != m + 1:
            raise ValueError(f"{what}: a signature batch must hold one item per (dealer, verifier) of the range")
        st = np.empty(m, dtype=np.uint8)
        keep += [msg, off, sig]
        args += [_ptr(msg), _ptr(off), _ptr(sig), _ptr(st)]
        outs.append(st)
    return args, outs, keep


class Context:
    """One kb_ctx: one CUDA device, one host thread (the reference is single-threaded)."""

    def __init__(self, device: int = 0):
        self.L = load_library()
        h = ctypes.c_void_p()
        rc = self.L.kb_ctx_create(device, ctypes.byref(h))
        if rc != 0:
            raise KBError(f"kb_ctx_create(device={device}) failed with {rc}: no usable CUDA device (there is no CPU fallback)")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.kb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise KBError(f"{what} failed with {rc}: {self.L.kb_last_error(self.h).decode(errors='replace')}")

    def wipe(self):
        self._check(self.L.kb_ctx_wipe(self.h), "kb_ctx_wipe")

    @property
    def sm_count(self):
        return self.L.kb_device_sm_count(self.h)

    @property
    def launches(self):
        return int(self.L.kb_launch_count(self.h))

    # ---- host-buffer API (numpy in / numpy out) ------------------------------------------
    def point_mul_base_batch(self, scalars, flags=0):
        s = _u8(scalars, (-1, 32))
        out = np.empty_like(s)
        self._check(self.L.kb_point_mul_base_batch(self.h, s.shape[0], _ptr(s), _ptr(out), flags), "kb_point_mul_base_batch")
        return out

    def point_mul_batch(self, scalars, points, flags=0):
        s = _u8(scalars, (-1, 32))
        p = _u8(points, (-1, 32))
        if p.shape[0] == 1 and s.shape[0] != 1:
            flags |= FLAG_SHARED_POINT
        out = np.empty_like(s)
        st = np.empty(s.shape[0], dtype=np.uint8)
        self._check(self.L.kb_point_mul_batch(self.h, s.shape[0], _ptr(s), _ptr(p), _ptr(out), _ptr(st), flags), "kb_point_mul_batch")
        return out, st

    def point_recode_batch(self, pts):
        p = _u8(pts, (-1, 32))
        out = np.empty_like(p)
        st = np.empty(p.shape[0], dtype=np.uint8)
        self._check(self.L.kb_point_recode_batch(self.h, p.shape[0], _ptr(p), _ptr(out), _ptr(st)), "kb_point_recode_batch")
        return out, st

    def point_from_limbs_batch(self, limbs):
        l = np.ascontiguousarray(limbs, dtype=np.int32).reshape(-1, 40)
        out = np.empty((l.shape[0], 32), dtype=np.uint8)
        self._check(self.L.kb_point_from_limbs_batch(self.h, l.shape[0], _ptr(l), _ptr(out)), "kb_point_from_limbs_batch")
        return out

    def point_add_batch(self, p, q, subtract=False):
        p = _u8(p, (-1, 32))
        q = _u8(q, (-1, 32))
        assert p.shape == q.shape
        out = np.empty_like(p)
        st = np.empty(p.shape[0], dtype=np.uint8)
        self._check(self.L.kb_point_add_batch(self.h, p.shape[0], _ptr(p), _ptr(q), _ptr(out), _ptr(st), int(subtract)), "kb_point_add_batch")
        return out, st

    def point_check_batch(self, pts):
        p = _u8(pts, (-1, 32))
        fl = np.empty(p.shape[0], dtype=np.uint8)
        self._check(self.L.kb_point_check_batch(self.h, p.shape[0], _ptr(p), _ptr(fl)), "kb_point_check_batch")
        return fl

    def point_decompress_batch(self, pts):
        """32-byte encodings -> (n, 32) uint32 words X, Y, Z, T (8 words each); status 1 = does not decode."""
        p = _u8(pts, (-1, 32))
        out = np.empty((p.shape[0], 32), dtype=np.uint32)
        st = np.empty(p.shape[0], dtype=np.uint8)
        self._check(self.L.kb_point_decompress_batch(self.h, p.shape[0], _ptr(p), _ptr(out), _ptr(st)), "kb_point_decompress_batch")
        return out, st

    def point_compress_batch(self, raw):
        r = np.ascontiguousarray(raw, dtype=np.uint32).reshape(-1, 32)
        out = np.empty((r.shape[0], 32), dtype=np.uint8)
        self._check(self.L.kb_point_compress_batch(self.h, r.shape[0], _ptr(r), _ptr(out)), "kb_point_compress_batch")
        return out

    def point_eq_batch(self, p, q):
        """Point::eq per pair: bit 0 = equal, bit 1 = an operand does not decode."""
        p, q = _u8(p, (-1, 32)), _u8(q, (-1, 32))
        if p.shape != q.shape:
            raise ValueError("point_eq_batch: operands must have the same number of points")
        out = np.empty(p.shape[0], dtype=np.uint8)
        self._check(self.L.kb_point_eq_batch(self.h, p.shape[0], _ptr(p), _ptr(q), _ptr(out)), "kb_point_eq_batch")
        return out

    def sc_reduce64_batch(self, digests):
        d = _u8(digests, (-1, 64))
        out = np.empty((d.shape[0], 32), dtype=np.uint8)
        self._check(self.L.kb_sc_reduce64_batch(self.h, d.shape[0], _ptr(d), _ptr(out)), "kb_sc_reduce64_batch")
        return out

    def sc_muladd_batch(self, a, b, c):
        a, b, c = _u8(a, (-1, 32)), _u8(b, (-1, 32)), _u8(c, (-1, 32))
        out = np.empty_like(a)
        self._check(self.L.kb_sc_muladd_batch(self.h, a.shape[0], _ptr(a), _ptr(b), _ptr(c), _ptr(out)), "kb_sc_muladd_batch")
        return out

    def sc_invert_batch(self, a):
        a = _u8(a, (-1, 32))
        out = np.empty_like(a)
        self._check(self.L.kb_sc_invert_batch(self.h, a.shape[0], _ptr(a), _ptr(out)), "kb_sc_invert_batch")
        return out

    def challenge_batch(self, r, a, msg, msg_off):
        r, a = _u8(r, (-1, 32)), _u8(a, (-1, 32))
        msg = _u8(msg)
        msg_off = np.ascontiguousarray(msg_off, dtype=np.uint64)
        out = np.empty_like(r)
        self._check(self.L.kb_challenge_batch(self.h, r.shape[0], _ptr(r), _ptr(a), _ptr(msg), _ptr(msg_off), _ptr(out)), "kb_challenge_batch")
        return out

    def verify_batch(self, pk, msg, msg_off, sig, schnorr=False, out=None):
        pk, sig = _u8(pk, (-1, 32)), _u8(sig, (-1, 64))
        msg = _u8(msg)
        msg_off = np.ascontiguousarray(msg_off, dtype=np.uint64)
        n = pk.shape[0]
        assert sig.shape[0] == n and msg_off.shape[0] == n + 1
        st = out if out is not None else np.empty(n, dtype=np.uint8)
        fn = self.L.kb_schnorr_verify_batch if schnorr else self.L.kb_eddsa_verify_batch
        self._check(fn(self.h, n, _ptr(pk), _ptr(msg), _ptr(msg_off), _ptr(sig), _ptr(st)), "kb_verify_batch")
        return st

    def eddsa_sign_batch(self, seeds, msg, msg_off):
        seeds = _u8(seeds, (-1, 32))
        msg = _u8(msg)
        msg_off = np.ascontiguousarray(msg_off, dtype=np.uint64)
        n = seeds.shape[0]
        sig = np.empty((n, 64), dtype=np.uint8)
        pk = np.empty((n, 32), dtype=np.uint8)
        self._check(self.L.kb_eddsa_sign_batch(self.h, n, _ptr(seeds), _ptr(msg), _ptr(msg_off), _ptr(sig), _ptr(pk)), "kb_eddsa_sign_batch")
        return sig, pk

    def pubpoly_eval_batch(self, commits, t, poly_id, idx):
        c = _u8(commits, (-1, 32))
        npoly = c.shape[0] // t
        assert npoly * t == c.shape[0]
        poly_id = np.ascontiguousarray(poly_id, dtype=np.uint32)
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        m = idx.shape[0]
        if poly_id.shape[0] != m:
            raise ValueError("pubpoly_eval_batch: poly_id and idx must have one entry per item")
        out = np.empty((m, 32), dtype=np.uint8)
        st = np.empty(m, dtype=np.uint8)
        self._check(self.L.kb_pubpoly_eval_batch(self.h, npoly, t, _ptr(c), m, _ptr(poly_id), _ptr(idx), _ptr(out), _ptr(st)), "kb_pubpoly_eval_batch")
        return out, st

    def vss_verify_deals_batch(self, commits, t, poly_id, idx, shares):
        c = _u8(commits, (-1, 32))
        npoly = c.shape[0] // t
        assert npoly * t == c.shape[0]
        poly_id = np.ascontiguousarray(poly_id, dtype=np.uint32)
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        sh = _u8(shares, (-1, 32))
        m = idx.shape[0]
        if poly_id.shape[0] != m or sh.shape[0] != m:
            raise ValueError("vss_verify_deals_batch: poly_id, idx and shares must have one row per item")
        verdict = np.empty(m, dtype=np.uint8)
        self._check(self.L.kb_vss_verify_deals_batch(self.h, npoly, t, _ptr(c), m, _ptr(poly_id), _ptr(idx), _ptr(sh), _ptr(verdict)), "kb_vss_verify_deals_batch")
        return verdict

    def dkg_verify_round(self, n, t, commits, shares, dealer_lo=0, dealer_hi=None, verdict=None, limbs=False):
        """commits: (ndealers*t, 32) uint8 encodings, or with limbs=True (ndealers*t, 40) int32 raw ref10 limbs."""
        c = np.ascontiguousarray(commits, dtype=np.int32).reshape(-1, 40) if limbs else _u8(commits, (-1, 32))
        sh = _u8(shares, (-1, 32))
        ndealers = c.shape[0] // t
        if ndealers * t != c.shape[0] or sh.shape[0] != ndealers * n:
            raise ValueError("dkg_verify_round: commits must hold ndealers*t points and shares ndealers*n scalars")
        if dealer_hi is None:
            dealer_hi = ndealers
        if not (0 <= dealer_lo <= dealer_hi <= ndealers):
            raise ValueError("dkg_verify_round: dealer range outside the commitments")
        if verdict is None:
            verdict = np.zeros(ndealers * n, dtype=np.uint8)
        if verdict.shape[0] != ndealers * n:
            raise ValueError("dkg_verify_round: verdict must hold ndealers*n bytes")
        fn = self.L.kb_dkg_verify_round_limbs if limbs else self.L.kb_dkg_verify_round
        self._check(fn(self.h, n, t, dealer_lo, dealer_hi, _ptr(c), _ptr(sh), _ptr(verdict)), "kb_dkg_verify_round")
        return verdict

    def pripoly_eval_batch(self, coeffs, t, n):
        """PriPoly::eval for every polynomial at indices 0..n-1: (npoly*n, 32) shares, polynomial-major."""
        c = _u8(coeffs, (-1, 32))
        npoly = c.shape[0] // t
        if npoly * t != c.shape[0]:
            raise ValueError("pripoly_eval_batch: coeffs must hold npoly*t scalars")
        out = np.empty((npoly * n, 32), dtype=np.uint8)
        self._check(self.L.kb_pripoly_eval_batch(self.h, npoly, t, _ptr(c), n, _ptr(out)), "kb_pripoly_eval_batch")
        return out

    def pubpoly_sum(self, commits, t):
        c = _u8(commits, (-1, 32))
        npoly = c.shape[0] // t
        assert npoly * t == c.shape[0]
        out = np.empty((t, 32), dtype=np.uint8)
        st = np.empty(t, dtype=np.uint8)
        self._check(self.L.kb_pubpoly_sum(self.h, npoly, t, _ptr(c), _ptr(out), _ptr(st)), "kb_pubpoly_sum")
        return out, st

    # ---- protocol-level operations ----------------------------------------------------------
    @staticmethod
    def _points(a, limbs):
        return np.ascontiguousarray(a, dtype=np.int32).reshape(-1, 40) if limbs else _u8(a, (-1, 32))

    def vss_session_ids(self, dealers, verifiers, commits, t, limbs=False):
        """session_id per dealer (vss/pedersen/vss.rs:1069): (ndealers,32) digests, (ndealers,) status."""
        d, v, c = self._points(dealers, limbs), self._points(verifiers, limbs), self._points(commits, limbs)
        nd = d.shape[0]
        if c.shape[0] != nd * t:
            raise ValueError("vss_session_ids: commits must hold ndealers*t points")
        out = np.empty((nd, 32), dtype=np.uint8)
        st = np.empty(nd, dtype=np.uint8)
        self._check(self.L.kb_vss_session_ids(self.h, nd, v.shape[0], t, int(limbs), _ptr(d), _ptr(v), _ptr(c), _ptr(out), _ptr(st)), "kb_vss_session_ids")
        return out, st

    def find_pub_batch(self, plist, queries, limbs=False):
        l, q = self._points(plist, limbs), self._points(queries, limbs)
        out = np.empty(q.shape[0], dtype=np.int32)
        self._check(self.L.kb_find_pub_batch(self.h, l.shape[0], _ptr(l), q.shape[0], _ptr(q), int(limbs), _ptr(out)), "kb_find_pub_batch")
        return out

    def dkg_process_round(self, n, t, commits, shares, deal=None, resp=None, dealer_lo=0, dealer_hi=None, limbs=False):
        """One deal-verification round: share checks + Schnorr verification of the deal and response signatures.
        deal / resp = (pk[m,32], msg flat, msg_off[m+1], sig[m,64]) for the m = (dealer_hi-dealer_lo)*n items, or None.
        Returns (verdict[ndealers*n], deal_status[m] | None, resp_status[m] | None)."""
        c = self._points(commits, limbs)
        sh = _u8(shares, (-1, 32))
        ndealers = c.shape[0] // t
        if dealer_hi is None:
            dealer_hi = ndealers
        if ndealers * t != c.shape[0] or sh.shape[0] != ndealers * n or not (0 <= dealer_lo <= dealer_hi <= ndealers):
            raise ValueError("dkg_process_round: inconsistent shapes")
        m = (dealer_hi - dealer_lo) * n
        verdict = np.zeros(ndealers * n, dtype=np.uint8)
        args, outs, keep = [], [], []
        for batch in (deal, resp):
            if batch is None:
                args += [None] * 5
                outs.append(None)
                continue
            pk, msg, off, sig = _u8(batch[0], (-1, 32)), _u8(batch[1]), np.ascontiguousarray(batch[2], dtype=np.uint64), _u8(batch[3], (-1, 64))
            if pk.shape[0] != m or sig.shape[0] != m or off.shape[0] != m + 1:
                raise ValueError("dkg_process_round: a signature batch must hold one item per (dealer, verifier) of the range")
            st = np.empty(m, dtype=np.uint8)
            keep += [pk, msg, off, sig]
            args += [_ptr(pk), _ptr(msg), _ptr(off), _ptr(sig), _ptr(st)]
            outs.append(st)
        self._check(self.L.kb_dkg_process_round(self.h, n, t, dealer_lo, dealer_hi, int(limbs), _ptr(c), _ptr(sh), _ptr(verdict), *args), "kb_dkg_process_round")
        return verdict, outs[0], outs[1]

    def dkg_process_round_keyed(self, n, t, commits, shares, dealers, verifiers=None, deal=None, resp=None, dealer_lo=0, dealer_hi=None, limbs=False):
        """dkg_process_round with the participants' keys as KeySets of this context: deal k is signed by dealer key
        dealer_lo + k // n, response k by verifier key k % n (verifiers=None: the dealers' set).
        deal / resp = (msg flat, msg_off[m+1], sig[m,64]) for the m = (dealer_hi-dealer_lo)*n items, or None."""
        if verifiers is None:
            verifiers = dealers
        c = self._points(commits, limbs)
        sh = _u8(shares, (-1, 32))
        ndealers = c.shape[0] // t
        if dealer_hi is None:
            dealer_hi = ndealers
        if ndealers * t != c.shape[0] or sh.shape[0] != ndealers * n or not (0 <= dealer_lo <= dealer_hi <= ndealers):
            raise ValueError("dkg_process_round_keyed: inconsistent shapes")
        verdict = np.zeros(ndealers * n, dtype=np.uint8)
        args, outs, keep = _keyed_batches(deal, resp, (dealer_hi - dealer_lo) * n, "dkg_process_round_keyed")
        self._check(self.L.kb_dkg_process_round_keyed(self.h, KeySet._h(dealers), KeySet._h(verifiers), n, t, dealer_lo, dealer_hi, int(limbs), _ptr(c), _ptr(sh), _ptr(verdict), *args),
                    "kb_dkg_process_round_keyed")
        return verdict, outs[0], outs[1]

    def vss_rabin_verify_deals_batch(self, commits, t, h_point, poly_id, idx, f_shares, g_shares):
        c = _u8(commits, (-1, 32))
        npoly = c.shape[0] // t
        hp = _u8(h_point, (32,))
        poly_id = np.ascontiguousarray(poly_id, dtype=np.uint32)
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        f, g = _u8(f_shares, (-1, 32)), _u8(g_shares, (-1, 32))
        m = idx.shape[0]
        if npoly * t != c.shape[0] or poly_id.shape[0] != m or f.shape[0] != m or g.shape[0] != m:
            raise ValueError("vss_rabin_verify_deals_batch: inconsistent shapes")
        verdict = np.empty(m, dtype=np.uint8)
        self._check(self.L.kb_vss_rabin_verify_deals_batch(self.h, npoly, t, _ptr(c), _ptr(hp), m, _ptr(poly_id), _ptr(idx), _ptr(f), _ptr(g), _ptr(verdict)), "kb_vss_rabin_verify_deals_batch")
        return verdict

    def dss_verify_partials(self, random_commits, long_commits, msg, idx, partials):
        """(verdict[m], hash scalar bytes) of DSS::process_partial_sig's group math for one signing session."""
        r, l = _u8(random_commits, (-1, 32)), _u8(long_commits, (-1, 32))
        if r.shape != l.shape:
            raise ValueError("dss_verify_partials: the two polynomials must have the same threshold")
        mb = _u8(np.frombuffer(bytes(msg), dtype=np.uint8)) if len(msg) else np.zeros(0, dtype=np.uint8)
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        p = _u8(partials, (-1, 32))
        m = idx.shape[0]
        if p.shape[0] != m:
            raise ValueError("dss_verify_partials: one partial per index")
        verdict = np.empty(m, dtype=np.uint8)
        hs = np.empty(32, dtype=np.uint8)
        self._check(self.L.kb_dss_verify_partials(self.h, r.shape[0], _ptr(r), _ptr(l), _ptr(mb) if mb.size else None, mb.size, m, _ptr(idx), _ptr(p), _ptr(verdict), _ptr(hs)), "kb_dss_verify_partials")
        return verdict, hs.tobytes()

    def recover_commit_batch(self, idx, points, ncols=1):
        """points: (ncols*k, 32) as [column][share]; returns (out[ncols,32], status[ncols])."""
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        p = _u8(points, (-1, 32))
        k = idx.shape[0]
        if p.shape[0] != ncols * k:
            raise ValueError("recover_commit_batch: points must hold ncols*k encodings")
        out = np.empty((ncols, 32), dtype=np.uint8)
        st = np.empty(ncols, dtype=np.uint8)
        self._check(self.L.kb_recover_commit_batch(self.h, ncols, k, _ptr(idx), _ptr(p), _ptr(out), _ptr(st)), "kb_recover_commit_batch")
        return out, st

    def recover_pub_poly(self, idx, points):
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        p = _u8(points, (-1, 32))
        k = idx.shape[0]
        if p.shape[0] != k:
            raise ValueError("recover_pub_poly: one point per index")
        out = np.empty((k, 32), dtype=np.uint8)
        st = np.empty(k, dtype=np.uint8)
        self._check(self.L.kb_recover_pub_poly(self.h, k, _ptr(idx), _ptr(p), _ptr(out), _ptr(st)), "kb_recover_pub_poly")
        return out, st

    def dkg_resharing_key(self, new_t, idx, coeffs, share_idx=0, share=None):
        """coeffs: (k*new_t, 32) as [qualified node][coefficient]; returns (commits[new_t,32], status[new_t], check | None)."""
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        c = _u8(coeffs, (-1, 32))
        k = idx.shape[0]
        if c.shape[0] != k * new_t:
            raise ValueError("dkg_resharing_key: coeffs must hold k*new_t encodings")
        out = np.empty((new_t, 32), dtype=np.uint8)
        st = np.empty(new_t, dtype=np.uint8)
        chk = np.zeros(1, dtype=np.uint8)
        sh = _u8(share, (32,)) if share is not None else None
        self._check(self.L.kb_dkg_resharing_key(self.h, new_t, k, _ptr(idx), _ptr(c), int(share_idx), _ptr(sh), _ptr(out), _ptr(st), _ptr(chk) if sh is not None else None), "kb_dkg_resharing_key")
        return out, st, (bool(chk[0]) if sh is not None else None)

    def msm(self, scalars, points, want_partial=False):
        s, p = _u8(scalars, (-1, 32)), _u8(points, (-1, 32))
        assert s.shape == p.shape
        out = np.empty(32, dtype=np.uint8)
        partial = np.empty(128, dtype=np.uint8)
        bad = np.zeros(1, dtype=np.uint64)
        self._check(self.L.kb_msm(self.h, s.shape[0], _ptr(s), _ptr(p), _ptr(out), _ptr(partial), _ptr(bad)), "kb_msm")
        if want_partial:
            return out.tobytes(), partial, int(bad[0])
        return out.tobytes(), int(bad[0])

    def point_sum(self, partials):
        p = _u8(partials, (-1, 128))
        out = np.empty(32, dtype=np.uint8)
        self._check(self.L.kb_point_sum(self.h, p.shape[0], _ptr(p), _ptr(out)), "kb_point_sum")
        return out.tobytes()

    def probe_imad(self, kind, iters):
        rate, ms = ctypes.c_double(), ctypes.c_double()
        self._check(self.L.kb_probe_imad(self.h, kind, iters, ctypes.byref(rate), ctypes.byref(ms)), "kb_probe_imad")
        return rate.value, ms.value

    def verify_kernel_timing(self, enable=True):
        """Switch per-kernel CUDA-event timing of dev_verify on or off."""
        self._check(self.L.kb_verify_kernel_times(self.h, 1 if enable else 0, None), "kb_verify_kernel_times")

    def last_verify_kernel_ms(self):
        """(first launch ms, second launch ms) of the most recent dev_verify; waits for it."""
        ms = (ctypes.c_float * 2)()
        self._check(self.L.kb_verify_kernel_times(self.h, 1, ms), "kb_verify_kernel_times")
        return float(ms[0]), float(ms[1])

    def keyset(self, pk):
        """Registers the public keys pk (nkeys x 32 encodings) for verification by key index (KeySet)."""
        return KeySet(self, pk)

    # ---- device-pointer API (torch CUDA tensors; enqueues on torch's current stream) --------
    @staticmethod
    def _dp(t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else None

    @staticmethod
    def _stream():
        import torch

        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def dev_verify(self, n, pk, msg, msg_off, sig, status, schnorr=False):
        self._check(self.L.kb_dev_eddsa_verify(self.h, n, self._dp(pk), self._dp(msg), self._dp(msg_off), self._dp(sig), self._dp(status), int(schnorr), self._stream()), "kb_dev_eddsa_verify")

    def dev_point_mul_base(self, n, scalars, out, flags=0):
        self._check(self.L.kb_dev_point_mul_base(self.h, n, self._dp(scalars), self._dp(out), flags, self._stream()), "kb_dev_point_mul_base")

    def dev_point_mul(self, n, scalars, points, out, status, flags=0):
        self._check(self.L.kb_dev_point_mul(self.h, n, self._dp(scalars), self._dp(points), self._dp(out), self._dp(status), flags, self._stream()), "kb_dev_point_mul")

    def dev_msm(self, n, scalars, points, out32, partial128, bad):
        self._check(self.L.kb_dev_msm(self.h, n, self._dp(scalars), self._dp(points), self._dp(out32), self._dp(partial128), self._dp(bad), self._stream()), "kb_dev_msm")

    def dev_msm_ext(self, n, scalars, points128, out32, partial128, bad):
        """MSM over points that are already decoded (128 bytes each: X, Y, Z, T words)."""
        self._check(self.L.kb_dev_msm_ext(self.h, n, self._dp(scalars), self._dp(points128), self._dp(out32), self._dp(partial128), self._dp(bad), self._stream()), "kb_dev_msm_ext")

    def dev_dkg_verify_round(self, n, t, ndealers, commits, shares, verdict, limbs=False):
        fn = self.L.kb_dev_dkg_verify_round_limbs if limbs else self.L.kb_dev_dkg_verify_round
        self._check(fn(self.h, n, t, ndealers, self._dp(commits), self._dp(shares), self._dp(verdict), self._stream()), "kb_dev_dkg_verify_round")

    def dev_dkg_process_round(self, n, t, ndealers, commits, shares, verdict, deal=None, resp=None, limbs=False):
        """deal / resp = (pk, msg, msg_off, sig, status) CUDA tensors or None."""
        a = []
        for batch in (deal, resp):
            a += [self._dp(x) for x in batch] if batch is not None else [None] * 5
        self._check(self.L.kb_dev_dkg_process_round(self.h, n, t, ndealers, int(limbs), self._dp(commits), self._dp(shares), self._dp(verdict), *a, self._stream()), "kb_dev_dkg_process_round")

    def dev_dkg_process_round_keyed(self, n, t, ndealers, commits, shares, verdict, dealers, verifiers=None, deal=None, resp=None, dealer_lo=0, limbs=False):
        """dkg_process_round_keyed on CUDA tensors for the ndealers dealers from dealer_lo on (the arrays start at the first
        of them); deal / resp = (msg, msg_off, sig, status) CUDA tensors or None."""
        if verifiers is None:
            verifiers = dealers
        a = []
        for batch in (deal, resp):
            a += [self._dp(x) for x in batch] if batch is not None else [None] * 4
        self._check(self.L.kb_dev_dkg_process_round_keyed(self.h, KeySet._h(dealers), KeySet._h(verifiers), n, t, dealer_lo, ndealers, int(limbs), self._dp(commits), self._dp(shares),
                                                          self._dp(verdict), *a, self._stream()), "kb_dev_dkg_process_round_keyed")

    def dev_pripoly_eval(self, npoly, t, coeffs, n, out):
        self._check(self.L.kb_dev_pripoly_eval(self.h, npoly, t, self._dp(coeffs), n, self._dp(out), self._stream()), "kb_dev_pripoly_eval")

    def dev_point_decompress(self, n, enc, out128, status):
        self._check(self.L.kb_dev_point_decompress(self.h, n, self._dp(enc), self._dp(out128), self._dp(status), self._stream()), "kb_dev_point_decompress")

    def dev_challenge(self, n, r32, a32, msg, msg_off, out32):
        self._check(self.L.kb_dev_challenge(self.h, n, self._dp(r32), self._dp(a32), self._dp(msg), self._dp(msg_off), self._dp(out32), self._stream()), "kb_dev_challenge")

    def dev_point_sum(self, k, partials, out32):
        self._check(self.L.kb_dev_point_sum(self.h, k, self._dp(partials), self._dp(out32), self._stream()), "kb_dev_point_sum")


class KeySet:
    """One kb_keyset: public keys registered with a Context, each with its comb on the device (384 KiB per key).
    Signatures then name their key by index; the statuses are those of Context.verify_batch with pk = keys[key_idx]."""

    def __init__(self, ctx: Context, pk):
        self.ctx = ctx   # the key set belongs to its context and must go before it
        self.L = ctx.L
        self.h = None
        p = _u8(pk, (-1, 32))
        self.nkeys = p.shape[0]
        h = ctypes.c_void_p()
        ctx._check(self.L.kb_keyset_create(ctx.h, self.nkeys, _ptr(p), ctypes.byref(h)), "kb_keyset_create")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.kb_keyset_destroy(self.h)
            self.h = None

    @staticmethod
    def _h(ks):
        return ks.h if ks is not None else None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def verify_batch(self, key_idx, msg, msg_off, sig, schnorr=False, out=None):
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        sig = _u8(sig, (-1, 64))
        msg = _u8(msg)
        msg_off = np.ascontiguousarray(msg_off, dtype=np.uint64)
        n = key_idx.shape[0]
        if sig.shape[0] != n or msg_off.shape[0] != n + 1:
            raise ValueError("KeySet.verify_batch: one key index and one signature per item, n+1 message offsets")
        st = out if out is not None else np.empty(n, dtype=np.uint8)
        self.ctx._check(self.L.kb_keyset_verify_batch(self.h, n, _ptr(key_idx), _ptr(msg), _ptr(msg_off), _ptr(sig), _ptr(st), int(schnorr)), "kb_keyset_verify_batch")
        return st

    def dev_verify(self, n, key_idx, msg, msg_off, sig, status, schnorr=False):
        """key_idx: n uint32 (torch int32 tensor), the rest as Context.dev_verify; an index outside the set gives status 0xFF."""
        dp = Context._dp
        self.ctx._check(self.L.kb_dev_keyset_verify(self.h, n, dp(key_idx), dp(msg), dp(msg_off), dp(sig), dp(status), int(schnorr), Context._stream()), "kb_dev_keyset_verify")

    def mul_batch(self, key_idx, scalars, flags=0):
        """(out, status) = Context.point_mul_batch(scalars, keys[key_idx], flags) byte for byte, from the keys' combs:
        Point::mul(s, Some(pk)) of dh_exchange.  flags: 0 or FLAG_VARTIME."""
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        s = _u8(scalars, (-1, 32))
        n = key_idx.shape[0]
        if s.shape[0] != n:
            raise ValueError("KeySet.mul_batch: one key index per scalar")
        out = np.empty_like(s)
        st = np.empty(n, dtype=np.uint8)
        self.ctx._check(self.L.kb_keyset_mul_batch(self.h, n, _ptr(key_idx), _ptr(s), _ptr(out), _ptr(st), flags), "kb_keyset_mul_batch")
        return out, st

    def dev_mul(self, n, key_idx, scalars, out, status, flags=0):
        """key_idx: n uint32 (torch int32 tensor), scalars / out n x 32 bytes, status n bytes (or None) on the device, on torch's
        current stream; an index outside the set gives status 0xFF and 32 zero bytes."""
        dp = Context._dp
        self.ctx._check(self.L.kb_dev_keyset_mul(self.h, n, dp(key_idx), dp(scalars), dp(out), dp(status), flags, Context._stream()), "kb_dev_keyset_mul")


class MultiContext:
    """One kb_mctx: the GPUs `devices` of this box driven from one process; every call takes the whole host batch."""

    def __init__(self, devices):
        self.L = load_library()
        devs = (ctypes.c_int * len(devices))(*devices)
        h = ctypes.c_void_p()
        rc = self.L.kb_mctx_create(devs, len(devices), ctypes.byref(h))
        if rc != 0:
            raise KBError(f"kb_mctx_create({list(devices)}) failed with {rc} (-2: no usable CUDA device, -4: NCCL); there is no CPU fallback")
        self.h = h
        self.devices = list(devices)

    def close(self):
        if getattr(self, "h", None):
            self.L.kb_mctx_destroy(self.h)
            self.h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise KBError(f"{what} failed with {rc}: {self.L.kb_mctx_last_error(self.h).decode(errors='replace')}")

    @property
    def launches(self):
        return int(self.L.kb_mctx_launch_count(self.h))

    def verify_batch(self, pk, msg, msg_off, sig, schnorr=False, out=None):
        pk, sig = _u8(pk, (-1, 32)), _u8(sig, (-1, 64))
        msg = _u8(msg)
        msg_off = np.ascontiguousarray(msg_off, dtype=np.uint64)
        n = pk.shape[0]
        assert sig.shape[0] == n and msg_off.shape[0] == n + 1
        st = out if out is not None else np.empty(n, dtype=np.uint8)
        self._check(self.L.kb_mctx_verify_batch(self.h, n, _ptr(pk), _ptr(msg), _ptr(msg_off), _ptr(sig), _ptr(st), int(schnorr)), "kb_mctx_verify_batch")
        return st

    def point_mul_base_batch(self, scalars, flags=0):
        s = _u8(scalars, (-1, 32))
        out = np.empty_like(s)
        self._check(self.L.kb_mctx_point_mul_base_batch(self.h, s.shape[0], _ptr(s), _ptr(out), flags), "kb_mctx_point_mul_base_batch")
        return out

    def point_mul_batch(self, scalars, points, flags=0):
        s, p = _u8(scalars, (-1, 32)), _u8(points, (-1, 32))
        if p.shape[0] == 1 and s.shape[0] != 1:
            flags |= FLAG_SHARED_POINT
        out = np.empty_like(s)
        st = np.empty(s.shape[0], dtype=np.uint8)
        self._check(self.L.kb_mctx_point_mul_batch(self.h, s.shape[0], _ptr(s), _ptr(p), _ptr(out), _ptr(st), flags), "kb_mctx_point_mul_batch")
        return out, st

    def dkg_process_round(self, n, t, commits, shares, deal=None, resp=None, limbs=False, verdict=None):
        c = Context._points(commits, limbs)
        sh = _u8(shares, (-1, 32))
        ndealers = c.shape[0] // t
        if ndealers * t != c.shape[0] or sh.shape[0] != ndealers * n:
            raise ValueError("dkg_process_round: inconsistent shapes")
        m = ndealers * n
        if verdict is None:
            verdict = np.zeros(m, dtype=np.uint8)
        args, outs, keep = [], [], []
        for batch in (deal, resp):
            if batch is None:
                args += [None] * 5
                outs.append(None)
                continue
            pk, msg, off, sig = _u8(batch[0], (-1, 32)), _u8(batch[1]), np.ascontiguousarray(batch[2], dtype=np.uint64), _u8(batch[3], (-1, 64))
            if pk.shape[0] != m or sig.shape[0] != m or off.shape[0] != m + 1:
                raise ValueError("dkg_process_round: a signature batch must hold one item per (dealer, verifier)")
            st = np.empty(m, dtype=np.uint8)
            keep += [pk, msg, off, sig]
            args += [_ptr(pk), _ptr(msg), _ptr(off), _ptr(sig), _ptr(st)]
            outs.append(st)
        self._check(self.L.kb_mctx_dkg_process_round(self.h, n, t, ndealers, int(limbs), _ptr(c), _ptr(sh), _ptr(verdict), *args), "kb_mctx_dkg_process_round")
        return verdict, outs[0], outs[1]

    def dkg_verify_round(self, n, t, commits, shares, limbs=False, verdict=None):
        return self.dkg_process_round(n, t, commits, shares, limbs=limbs, verdict=verdict)[0]

    def keyset(self, pk):
        """Registers the public keys pk (nkeys x 32 encodings) on every device of this context (MultiKeySet)."""
        return MultiKeySet(self, pk)

    def dkg_process_round_keyed(self, n, t, commits, shares, dealers, verifiers=None, deal=None, resp=None, limbs=False, verdict=None):
        """dkg_process_round with the participants' keys as MultiKeySets of this context, split by dealer: deal k is
        signed by dealer key k // n, response k by verifier key k % n (verifiers=None: the dealers' set).
        deal / resp = (msg flat, msg_off[m+1], sig[m,64]) for the m = ndealers*n items, or None."""
        if verifiers is None:
            verifiers = dealers
        c = Context._points(commits, limbs)
        sh = _u8(shares, (-1, 32))
        ndealers = c.shape[0] // t
        if ndealers * t != c.shape[0] or sh.shape[0] != ndealers * n:
            raise ValueError("dkg_process_round_keyed: inconsistent shapes")
        if verdict is None:
            verdict = np.zeros(ndealers * n, dtype=np.uint8)
        args, outs, keep = _keyed_batches(deal, resp, ndealers * n, "dkg_process_round_keyed")
        self._check(self.L.kb_mctx_dkg_process_round_keyed(self.h, KeySet._h(dealers), KeySet._h(verifiers), n, t, ndealers, int(limbs), _ptr(c), _ptr(sh), _ptr(verdict), *args),
                    "kb_mctx_dkg_process_round_keyed")
        return verdict, outs[0], outs[1]

    def msm(self, scalars, points):
        s, p = _u8(scalars, (-1, 32)), _u8(points, (-1, 32))
        assert s.shape == p.shape
        out = np.empty(32, dtype=np.uint8)
        bad = np.zeros(1, dtype=np.uint64)
        self._check(self.L.kb_mctx_msm(self.h, s.shape[0], _ptr(s), _ptr(p), _ptr(out), _ptr(bad)), "kb_mctx_msm")
        return out.tobytes(), int(bad[0])


class MultiKeySet:
    """One kb_mkeyset: public keys registered on every device of a MultiContext.  Each device holds every key
    (384 KiB per key on each GPU); verify_batch splits a batch by index like MultiContext.verify_batch."""

    def __init__(self, mctx: MultiContext, pk):
        self.mctx = mctx   # the key set belongs to its context and must go before it
        self.L = mctx.L
        self.h = None
        p = _u8(pk, (-1, 32))
        self.nkeys = p.shape[0]
        h = ctypes.c_void_p()
        mctx._check(self.L.kb_mctx_keyset_create(mctx.h, self.nkeys, _ptr(p), ctypes.byref(h)), "kb_mctx_keyset_create")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.kb_mctx_keyset_destroy(self.h)
            self.h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def verify_batch(self, key_idx, msg, msg_off, sig, schnorr=False, out=None):
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        sig = _u8(sig, (-1, 64))
        msg = _u8(msg)
        msg_off = np.ascontiguousarray(msg_off, dtype=np.uint64)
        n = key_idx.shape[0]
        if sig.shape[0] != n or msg_off.shape[0] != n + 1:
            raise ValueError("MultiKeySet.verify_batch: one key index and one signature per item, n+1 message offsets")
        st = out if out is not None else np.empty(n, dtype=np.uint8)
        self.mctx._check(self.L.kb_mctx_keyset_verify_batch(self.h, n, _ptr(key_idx), _ptr(msg), _ptr(msg_off), _ptr(sig), _ptr(st), int(schnorr)), "kb_mctx_keyset_verify_batch")
        return st

    def mul_batch(self, key_idx, scalars, flags=0):
        """KeySet.mul_batch split by index over the devices."""
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        s = _u8(scalars, (-1, 32))
        n = key_idx.shape[0]
        if s.shape[0] != n:
            raise ValueError("MultiKeySet.mul_batch: one key index per scalar")
        out = np.empty_like(s)
        st = np.empty(n, dtype=np.uint8)
        self.mctx._check(self.L.kb_mctx_keyset_mul_batch(self.h, n, _ptr(key_idx), _ptr(s), _ptr(out), _ptr(st), flags), "kb_mctx_keyset_mul_batch")
        return out, st
