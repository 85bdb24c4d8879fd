"""Verification by public-key bytes under a key set, against the two calls a caller would otherwise make.

2^20 signatures over 64-byte messages, 1/64 spoiled in bench.spoil's nine classes.  An item's signer is a registered key
with probability `hit` (random positions), otherwise one of 4096 unregistered keys.  For hit fractions below 1 the set
holds the K keys; for hit = 1 it also holds the invalid keys spoil writes, so that every item hits and
kb_dev_keyset_verify can be given the index array a caller would have built.  Timed by CUDA events on one stream,
median of --reps runs after warm-up, the calls alternating on the same inputs; every status of every run is checked
against kb_dev_eddsa_verify's and the hit count against the host's; any mismatch exits non-zero.

  kb_dev_keyset_verify_pk  vs  kb_dev_eddsa_verify (every fraction)  and  kb_dev_keyset_verify (hit = 1)

The host forms (host clock around the call, which returns after its copies) are timed at K = 1 024:
kb_keyset_verify_pk_batch (plain staging, one copy in and out) against kb_eddsa_verify_batch (pipelined chunks) and,
at hit = 1, kb_keyset_verify_batch.  One JSON line on stdout (and in --out) with the GPU's name, power limit and max SM
clock read in the same run.

  python tools/bench_keyset_pk.py [--reps 7] [--out profiles/r8_bench_keyset_pk.json]
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

N = 1 << 20
FRACS = {"0": 0.0, "1/2": 0.5, "63/64": 63 / 64, "1": 1.0}


def scalars(tag, n):
    a = bench.xof(tag, 32 * n).reshape(n, 32).copy()
    a[:, 31] &= 0x0F
    return a


def rows(a):
    a = np.ascontiguousarray(a)
    return a.view(np.dtype((np.void, 32))).reshape(-1)


def make_batch(ctx, nkeys, hit):
    """(set keys, pk, msg, off, sig, key_idx of every item in the set keys or None)"""
    rng = np.random.default_rng(nkeys)
    a_reg = scalars(f"kyber-b200/keyset_pk/keys/{nkeys}", nkeys)
    keys = ctx.point_mul_base_batch(a_reg)
    a_un = scalars("kyber-b200/keyset_pk/others", 4096)
    keys_un = ctx.point_mul_base_batch(a_un)
    is_hit = np.zeros(N, dtype=bool)
    is_hit[rng.permutation(N)[: round(N * hit)]] = True
    ki, ku = rng.integers(0, nkeys, size=N), rng.integers(0, 4096, size=N)
    a = np.where(is_hit[:, None], a_reg[ki], a_un[ku])
    pk = np.where(is_hit[:, None], keys[ki], keys_un[ku])
    r = scalars(f"kyber-b200/keyset_pk/nonces/{nkeys}", N)
    msg = bench.xof(f"kyber-b200/keyset_pk/msgs/{nkeys}", 64 * N).copy()
    off = np.arange(N + 1, dtype=np.uint64) * np.uint64(64)
    R = ctx.point_mul_base_batch(r)
    sig = np.concatenate([R, ctx.sc_muladd_batch(ctx.challenge_batch(R, pk, msg, off), a, r)], axis=1)
    bench.spoil(pk, msg, sig, 0, N)
    key_idx = None
    if hit == 1.0:
        keys, inv = np.unique(pk, axis=0, return_inverse=True)
        key_idx = inv.reshape(-1).astype(np.uint32)
    return keys, pk, msg, off, sig, key_idx


def run(kb, ctx, nkeys, frac, reps, host):
    dev = torch.device("cuda", 0)
    keys, pk, msg, off, sig, key_idx = make_batch(ctx, nkeys, FRACS[frac])
    hits_host = int(np.isin(rows(pk), rows(keys)).sum())
    ks = ctx.keyset(keys)
    d_pk, d_sig, d_msg = (torch.from_numpy(x).to(dev) for x in (pk, sig, msg))
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    st = {k: torch.full((N,), 99, dtype=torch.uint8, device=dev) for k in ("pk", "general", "keyset")}
    d_hits = torch.zeros(1, dtype=torch.int64, device=dev)
    calls = {"pk": lambda: ks.dev_verify_pk(N, d_pk, d_msg, d_off, d_sig, st["pk"], hits=d_hits),
             "general": lambda: ctx.dev_verify(N, d_pk, d_msg, d_off, d_sig, st["general"])}
    if key_idx is not None:
        d_idx = torch.from_numpy(key_idx.view(np.int32)).to(dev)
        calls["keyset"] = lambda: ks.dev_verify(N, d_idx, d_msg, d_off, d_sig, st["keyset"])
    for _ in range(2):
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    mism = 0
    for _ in range(reps):
        for label, fn in calls.items():
            st[label].fill_(99)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[label].append(e0.elapsed_time(e1))
        ref = st["general"].cpu()
        mism += sum(int((st[k].cpu() != ref).sum()) for k in calls if k != "general")
        mism += int(int(d_hits.cpu()[0]) != hits_host)
    out = {"keys": int(nkeys), "set_keys": int(keys.shape[0]), "hit_fraction": frac, "hits": hits_host,
           **{f"{k}_ms": statistics.median(v) for k, v in times.items()}, **{f"{k}_ms_all": v for k, v in times.items()}}
    out["pk_over_general"] = out["pk_ms"] / out["general_ms"]
    if "keyset_ms" in out:
        out["pk_over_keyset"] = out["pk_ms"] / out["keyset_ms"]
    if host:
        want = ctx.verify_batch(pk, msg, off, sig)
        hcalls = {"pk_host": lambda: ks.verify_pk_batch(pk, msg, off, sig, return_hits=True)[0], "general_host": lambda: ctx.verify_batch(pk, msg, off, sig)}
        if key_idx is not None:
            hcalls["keyset_host"] = lambda: ks.verify_batch(key_idx, msg, off, sig)
        ht = {k: [] for k in hcalls}
        for fn in hcalls.values():
            fn()
        for _ in range(reps):
            for label, fn in hcalls.items():
                t0 = time.perf_counter()
                got = fn()
                ht[label].append((time.perf_counter() - t0) * 1e3)
                mism += int((got != want).sum())
        out.update({f"{k}_ms": statistics.median(v) for k, v in ht.items()})
    out["status_mismatches"] = mism
    ks.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--keys", type=str, default="1024,65536")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if a.reps < 5:
        sys.exit("--reps must be at least 5")
    if not torch.cuda.is_available():
        sys.exit("bench_keyset_pk: no CUDA device (there is no CPU path)")
    kb = importlib.import_module("kyber-rs_b200")
    ctx = kb.Context(0)
    res = {"metric": "verify by pk bytes under a key set vs the general verifier and the index-array key-set call, CUDA-event ms per 2^20 EdDSA signatures (median)",
           **gpu_info(), "reps": a.reps, "configs": {}}
    for k in (int(x) for x in a.keys.split(",") if x):
        for frac in FRACS:
            c = run(kb, ctx, k, frac, a.reps, host=(k == 1024))
            res["configs"][f"K={k},hit={frac}"] = c
            print(f"K={k} hit={frac}: pk {c['pk_ms']:.3f} ms, general {c['general_ms']:.3f} ms" + (f", keyset {c['keyset_ms']:.3f} ms" if "keyset_ms" in c else "")
                  + (f"; host pk {c['pk_host_ms']:.1f} ms, general {c['general_host_ms']:.1f} ms" if "pk_host_ms" in c else ""), file=sys.stderr)
    ok = all(c["status_mismatches"] == 0 for c in res["configs"].values())
    res["all_statuses_equal"] = ok
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
