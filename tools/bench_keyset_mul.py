"""Keyed scalar multiplication (kb_dev_keyset_mul) against the general one (kb_dev_point_mul with points = keys[key_idx]), on
the same inputs.

For each configuration, 2^20 random 32-byte scalars are multiplied by K registered keys: K = 1, 1024 and 65536 with random
key_idx, and the shape of a batched deal round, 1024 keys with item k using key k % 1024 (the n^2 Diffie-Hellman steps of
encrypted_deal).  Each runs with flags 0 (secret scalars, constant-time select) and KB_FLAG_VARTIME.  The tool times both
calls by CUDA events on one stream (median of --reps runs after warm-up, the two calls alternating) and compares their
outputs and statuses item by item after every timed pair; any mismatch exits non-zero.  Table traffic is counted from the
shapes: the constant-time select reads 8 comb entries of 96 bytes per window, 64 windows per item; the public-scalar
select reads at most one.  One JSON line on stdout (and in --out), with the GPU's name, power limit and max SM clock read in
the same run.

  python tools/bench_keyset_mul.py [--reps 7] [--out profiles/r5_bench_keyset_mul.json]
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
ENTRY_BYTES = 96


def run_config(ctx, name, nkeys, key_idx, flags, reps):
    dev = torch.device("cuda", 0)
    n = key_idx.shape[0]
    tag = f"kyber-b200/keyset-mul/{name}"
    keys = ctx.point_mul_base_batch(bench.xof(tag + "/keys", 32 * nkeys).reshape(nkeys, 32), 1)
    scalars = bench.xof(tag + f"/scalars/{flags}", 32 * n).reshape(n, 32)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ks = ctx.keyset(keys)
    build_ms = (time.perf_counter() - t0) * 1e3
    d_idx = torch.from_numpy(key_idx.view(np.int32)).to(dev)
    d_s = torch.from_numpy(scalars.copy()).to(dev)
    d_pts = torch.from_numpy(keys[key_idx]).to(dev)
    outs = {lab: (torch.empty((n, 32), dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)) for lab in ("keyset", "general")}

    def keyed():
        ks.dev_mul(n, d_idx, d_s, *outs["keyset"], flags=flags)

    def general():
        ctx.dev_point_mul(n, d_s, d_pts, *outs["general"], flags)

    for _ in range(2):
        keyed()
        general()
    torch.cuda.synchronize()
    times = {"keyset": [], "general": []}
    mism = 0
    for _ in range(reps):
        for lab in ("keyset", "general"):
            outs[lab][0].fill_(0xAA)
            outs[lab][1].fill_(99)
        for label, fn in (("keyset", keyed), ("general", general)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[label].append(e0.elapsed_time(e1))
        (ok, sk), (og, sg) = outs["keyset"], outs["general"]
        mism += int(((ok != og).any(dim=1) | (sk != sg)).sum().item())
    bad_status = int((outs["general"][1] != 0).sum().item())
    ks.close()
    mk, mg = statistics.median(times["keyset"]), statistics.median(times["general"])
    table_bytes = n * 64 * (8 if flags == 0 else 1) * ENTRY_BYTES
    return {
        "n": n, "keys": int(nkeys), "flags": int(flags),
        "keyset_ms": mk, "general_ms": mg, "speedup": mg / mk,
        "keyset_muls_per_s": n / (mk * 1e-3), "general_muls_per_s": n / (mg * 1e-3),
        "keyset_ms_all": times["keyset"], "general_ms_all": times["general"],
        "table_bytes_read": table_bytes, "table_read_GB_per_s": table_bytes / (mk * 1e-3) / 1e9,
        "build_ms": build_ms, "comb_bytes": int(nkeys) * 393216,
        "mismatches": mism, "nonzero_status": bad_status,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--keys", type=str, default="1,1024,65536")
    ap.add_argument("--no-deal", action="store_true")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if a.reps < 7:
        sys.exit("--reps must be at least 7")
    if not torch.cuda.is_available():
        sys.exit("bench_keyset_mul: no CUDA device (there is no CPU path)")
    kb = importlib.import_module("kyber-rs_b200")
    ctx = kb.Context(0)
    n = 1 << LOG2N
    rng = np.random.default_rng(2026)
    res = {"metric": "keyed vs general scalar multiplication, CUDA-event ms per 2^20 items (median)", **gpu_info(), "reps": a.reps, "configs": {}}
    shapes = [(f"K={k}", k, rng.integers(0, k, size=n, dtype=np.uint32)) for k in (int(x) for x in a.keys.split(",") if x)]
    if not a.no_deal:
        shapes.append(("deal_1024", 1024, (np.arange(n) % 1024).astype(np.uint32)))
    for label, k, key_idx in shapes:
        for flags in (0, kb.FLAG_VARTIME):
            name = f"{label}/{'vartime' if flags else 'ct'}"
            c = res["configs"][name] = run_config(ctx, label, k, key_idx, flags, a.reps)
            print(f"{name}: {c['keyset_ms']:.3f} ms vs {c['general_ms']:.3f} ms (x{c['speedup']:.2f}), mismatches {c['mismatches']}", file=sys.stderr)
    ok = all(c["mismatches"] == 0 and c["nonzero_status"] == 0 for c in res["configs"].values())
    res["all_outputs_equal"] = ok
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
