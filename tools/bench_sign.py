"""Signing rates: kb_schnorr_sign_batch against the four-call composition it replaces, Schnorr signer sets against
kb_schnorr_sign_batch, and an EdDSA signer set against kb_eddsa_sign_batch, on the same inputs.

2^20 signatures over 64-byte messages.  Device buffers: CUDA events on one stream around kb_dev_schnorr_sign, around
kb_dev_signerset_sign, and around the device part of the composition (two constant-time kb_dev_point_mul_base calls and
kb_dev_challenge; its sc_muladd step has no device form, so that figure leaves it out).  Host buffers: a host clock around
each blocking call (each ends in a device synchronisation): kb_schnorr_sign_batch, the composition as the four host calls
point_mul_base x2 / challenge / sc_muladd, kb_signerset_sign_batch and kb_eddsa_sign_batch.  Signer sets run at K = 1, 1024
and 65536 keys with random key_idx.  Median of --reps runs after warm-up, the compared calls alternating; every output is
compared byte for byte with its reference after every timed pair, and any mismatch exits non-zero.  One JSON line on
stdout (and in --out), with the GPU's name, power limit and max SM clock read in the same run.

  python tools/bench_sign.py [--reps 7] [--out profiles/r7_bench_sign.json]
"""
import argparse
import importlib
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_keyset import gpu_info  # noqa: E402

LOG2N = 20
MSG_LEN = 64


def _ev_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def _host_ms(fn):
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def _timed(fns, reps, check):
    """fns: {label: (kind, fn)} with kind 'dev' (CUDA events) or 'host' (host clock); check() after every round -> mismatches"""
    for _ in range(2):
        for _, fn in fns.values():
            fn()
    torch.cuda.synchronize()
    times = {lab: [] for lab in fns}
    mism = 0
    for _ in range(reps):
        for lab, (kind, fn) in fns.items():
            times[lab].append(_ev_ms(fn) if kind == "dev" else _host_ms(fn)[0])
        mism += check()
    return {lab: statistics.median(t) for lab, t in times.items()}, {lab + "_all": t for lab, t in times.items()}, mism


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--keys", type=str, default="1,1024,65536")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if a.reps < 7:
        sys.exit("--reps must be at least 7")
    if not torch.cuda.is_available():
        sys.exit("bench_sign: no CUDA device (there is no CPU path)")
    kb = importlib.import_module("kyber-rs_b200")
    ctx = kb.Context(0)
    dev = torch.device("cuda", 0)
    n = 1 << LOG2N
    res = {"metric": "signing, ms per 2^20 signatures over 64-byte messages (median)", **gpu_info(), "reps": a.reps, "n": n, "configs": {}}
    flat = bench.xof("kyber-b200/sign/msgs", MSG_LEN * n)
    off = (np.arange(n + 1, dtype=np.uint64) * MSG_LEN)
    k = bench.xof("kyber-b200/sign/nonces", 32 * n).reshape(n, 32).copy()
    k[:, 31] &= 0x0F
    d_m, d_off, d_k = (torch.from_numpy(flat.copy()).to(dev), torch.from_numpy(off.view(np.int64)).to(dev), torch.from_numpy(k).to(dev))
    rng = np.random.default_rng(2026)
    ok = True

    # ---- kb_schnorr_sign_batch against the composition, secrets all distinct
    x = bench.xof("kyber-b200/sign/secrets", 32 * n).reshape(n, 32).copy()
    x[:, 31] &= 0x0F
    d_x = torch.from_numpy(x).to(dev)
    bufs = {lab: torch.empty((n, 64), dtype=torch.uint8, device=dev) for lab in ("fused", "comp")}
    d_pk, d_r, d_h = (torch.empty((n, 32), dtype=torch.uint8, device=dev) for _ in range(3))
    host_out = {}

    def comp_host():
        A = ctx.point_mul_base_batch(x)
        R = ctx.point_mul_base_batch(k)
        h = ctx.challenge_batch(R, A, flat, off)
        return np.concatenate([R, ctx.sc_muladd_batch(x, h, k)], axis=1)

    def comp_dev():
        ctx.dev_point_mul_base(n, d_x, d_pk)
        ctx.dev_point_mul_base(n, d_k, d_r)
        ctx.dev_challenge(n, d_r, d_pk, d_m, d_off, d_h)

    def check_fused():
        host_out["fused"] = ctx.schnorr_sign_batch(x, k, flat, off)[0]
        host_out["comp"] = comp_host()
        bad = int((host_out["fused"] != host_out["comp"]).any(axis=1).sum())
        torch.cuda.synchronize()
        bad += int((bufs["fused"].cpu().numpy() != host_out["comp"]).any(axis=1).sum())
        bad += int((d_r.cpu().numpy() != host_out["comp"][:, :32]).any(axis=1).sum())
        return bad

    med, alls, mism = _timed({
        "fused_dev_ms": ("dev", lambda: ctx.dev_schnorr_sign(n, d_x, d_k, d_m, d_off, bufs["fused"], d_pk)),
        "composition_dev_without_muladd_ms": ("dev", comp_dev),
        "fused_host_ms": ("host", lambda: ctx.schnorr_sign_batch(x, k, flat, off)),
        "composition_host_ms": ("host", comp_host),
    }, a.reps, check_fused)
    c = res["configs"]["schnorr_sign_batch"] = {**med, **alls, "mismatches": mism,
                                                "fused_dev_sigs_per_s": n / (med["fused_dev_ms"] * 1e-3), "fused_host_sigs_per_s": n / (med["fused_host_ms"] * 1e-3),
                                                "composition_host_sigs_per_s": n / (med["composition_host_ms"] * 1e-3)}
    ok &= mism == 0
    print(f"schnorr_sign_batch: dev {med['fused_dev_ms']:.3f} ms (composition w/o muladd {med['composition_dev_without_muladd_ms']:.3f}), "
          f"host {med['fused_host_ms']:.3f} ms vs {med['composition_host_ms']:.3f} ms, mismatches {mism}", file=sys.stderr)
    del d_x, bufs

    # ---- Schnorr signer sets against kb_schnorr_sign_batch on secrets[key_idx]
    for nkeys in (int(v) for v in a.keys.split(",") if v):
        keys = bench.xof(f"kyber-b200/sign/set-keys/{nkeys}", 32 * nkeys).reshape(nkeys, 32).copy()
        keys[:, 31] &= 0x0F
        key_idx = rng.integers(0, nkeys, size=n, dtype=np.uint32)
        xs = keys[key_idx]
        d_xs, d_idx = torch.from_numpy(xs).to(dev), torch.from_numpy(key_idx.view(np.int32)).to(dev)
        d_sig = {lab: torch.empty((n, 64), dtype=torch.uint8, device=dev) for lab in ("set", "fused")}
        t0 = time.perf_counter()
        ss = ctx.signerset(keys)
        build_ms = (time.perf_counter() - t0) * 1e3

        def check_set():
            want = ctx.schnorr_sign_batch(xs, k, flat, off)[0]
            torch.cuda.synchronize()
            bad = int((ss.sign_batch(key_idx, flat, off, k) != want).any(axis=1).sum())
            bad += int((d_sig["set"].cpu().numpy() != want).any(axis=1).sum()) + int((d_sig["fused"].cpu().numpy() != want).any(axis=1).sum())
            return bad

        med, alls, mism = _timed({
            "set_dev_ms": ("dev", lambda: ss.dev_sign(n, d_idx, d_k, d_m, d_off, d_sig["set"])),
            "fused_dev_ms": ("dev", lambda: ctx.dev_schnorr_sign(n, d_xs, d_k, d_m, d_off, d_sig["fused"], None)),
            "set_host_ms": ("host", lambda: ss.sign_batch(key_idx, flat, off, k)),
            "fused_host_ms": ("host", lambda: ctx.schnorr_sign_batch(xs, k, flat, off)),
        }, a.reps, check_set)
        ss.close()
        res["configs"][f"schnorr_set_K={nkeys}"] = {**med, **alls, "keys": nkeys, "build_ms": build_ms, "set_bytes": 64 * nkeys, "mismatches": mism,
                                                    "dev_speedup": med["fused_dev_ms"] / med["set_dev_ms"], "host_speedup": med["fused_host_ms"] / med["set_host_ms"],
                                                    "set_dev_sigs_per_s": n / (med["set_dev_ms"] * 1e-3)}
        ok &= mism == 0
        print(f"schnorr set K={nkeys}: dev {med['set_dev_ms']:.3f} vs {med['fused_dev_ms']:.3f} ms, host {med['set_host_ms']:.3f} vs {med['fused_host_ms']:.3f} ms, "
              f"mismatches {mism}", file=sys.stderr)
        del d_xs, d_idx, d_sig

    # ---- EdDSA: kb_eddsa_sign_batch (host buffers only) against an EdDSA signer set
    nkeys = 1024
    seeds = bench.xof("kyber-b200/sign/eddsa-seeds", 32 * nkeys).reshape(nkeys, 32).copy()
    key_idx = rng.integers(0, nkeys, size=n, dtype=np.uint32)
    sd = seeds[key_idx]
    d_idx = torch.from_numpy(key_idx.view(np.int32)).to(dev)
    d_sig = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    es = ctx.signerset(seeds, kb.SIGNER_EDDSA)

    def check_eddsa():
        want = ctx.eddsa_sign_batch(sd, flat, off)[0]
        torch.cuda.synchronize()
        return int((es.sign_batch(key_idx, flat, off) != want).any(axis=1).sum()) + int((d_sig.cpu().numpy() != want).any(axis=1).sum())

    med, alls, mism = _timed({
        "set_dev_ms": ("dev", lambda: es.dev_sign(n, d_idx, None, d_m, d_off, d_sig)),
        "set_host_ms": ("host", lambda: es.sign_batch(key_idx, flat, off)),
        "eddsa_sign_batch_host_ms": ("host", lambda: ctx.eddsa_sign_batch(sd, flat, off)),
    }, a.reps, check_eddsa)
    es.close()
    res["configs"]["eddsa_set_K=1024"] = {**med, **alls, "keys": nkeys, "mismatches": mism, "host_speedup": med["eddsa_sign_batch_host_ms"] / med["set_host_ms"],
                                          "set_dev_sigs_per_s": n / (med["set_dev_ms"] * 1e-3)}
    ok &= mism == 0
    print(f"eddsa set K=1024: dev {med['set_dev_ms']:.3f} ms, host {med['set_host_ms']:.3f} vs kb_eddsa_sign_batch {med['eddsa_sign_batch_host_ms']:.3f} ms, mismatches {mism}",
          file=sys.stderr)

    res["all_outputs_equal"] = bool(ok)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ctx.close()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
