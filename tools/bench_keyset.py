"""Key sets against the general verifier, on the same inputs.

For each configuration, 2^20 signatures with 64-byte messages are made under K keys (random key_idx), and the nine
invalid classes of bench.spoil are applied; a class that alters pk turns that pk into an extra, invalid key of the set.
The tool then times, by CUDA events on one stream (median of --reps runs after warm-up, alternating the two calls),
kb_dev_keyset_verify(keys, key_idx) and kb_dev_eddsa_verify(pk = keys[key_idx]), and compares their statuses item by
item; any mismatch exits non-zero.  Configurations: K = 1, 1024, 65536 (EdDSA) and the DKG shape, 1024 keys x 1024
Schnorr signatures each (dealer-major).  The key-set build is timed on the host around kb_keyset_create (which waits
for the build).  One JSON line on stdout (and in --out), with the GPU's name, power limit and max SM clock read in
the same run.

  python tools/bench_keyset.py [--reps 7] [--out profiles/r3_bench_keyset.json]
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

LOG2N = 20


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # pragma: no cover
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": None, "max_sm_clock": None, "nvidia_smi": str(e)}


def make_config(ctx, name, nkeys, key_idx):
    """Keys, signatures (signed with the library's own primitives, as bench.make_batch), spoiled items; returns
    (keys incl. the extra invalid ones, key_idx, pk per item, msg, off, sig, expected EdDSA statuses)."""
    n = key_idx.shape[0]
    tag = f"kyber-b200/keyset/{name}"
    a = bench.xof(tag + "/keys", 32 * nkeys).reshape(nkeys, 32).copy()
    a[:, 0] &= 0xF8
    a[:, 31] &= 0x7F
    a[:, 31] |= 0x40
    r = bench.xof(tag + "/nonces", 32 * n).reshape(n, 32).copy()
    r[:, 31] &= 0x0F
    msg = bench.xof(tag + "/msgs", 64 * n).copy()
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(64)
    keys = ctx.point_mul_base_batch(a)
    pk = keys[key_idx]
    R = ctx.point_mul_base_batch(r)
    h = ctx.challenge_batch(R, pk, msg, off)
    s = ctx.sc_muladd_batch(h, a[key_idx], r)
    sig = np.concatenate([R, s], axis=1)
    expect = bench.spoil(pk, msg, sig, 0, n)
    # altered keys become extra keys of the set
    changed = np.nonzero((pk != keys[key_idx]).any(axis=1))[0]
    extra, inv = np.unique(pk[changed], axis=0, return_inverse=True)
    key_idx = key_idx.copy()
    key_idx[changed] = nkeys + inv.reshape(-1).astype(np.uint32)
    keys = np.concatenate([keys, extra])
    assert (keys[key_idx] == pk).all()
    return keys, key_idx, pk, msg, off, sig, expect


def run_config(kb, ctx, name, nkeys, key_idx, schnorr, reps):
    dev = torch.device("cuda", 0)
    keys, key_idx, pk, msg, off, sig, expect = make_config(ctx, name, nkeys, key_idx)
    n = key_idx.shape[0]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ks = ctx.keyset(keys)
    build_ms = (time.perf_counter() - t0) * 1e3
    d_idx = torch.from_numpy(key_idx.view(np.int32)).to(dev)
    d_pk, d_sig, d_msg = (torch.from_numpy(x).to(dev) for x in (pk, sig, msg))
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    d_st_k = torch.full((n,), 99, dtype=torch.uint8, device=dev)
    d_st_g = torch.full((n,), 99, dtype=torch.uint8, device=dev)

    def keyed():
        ks.dev_verify(n, d_idx, d_msg, d_off, d_sig, d_st_k, schnorr=schnorr)

    def general():
        ctx.dev_verify(n, d_pk, d_msg, d_off, d_sig, d_st_g, schnorr=schnorr)

    for _ in range(2):
        keyed()
        general()
    torch.cuda.synchronize()
    times = {"keyset": [], "general": []}
    for _ in range(reps):
        for label, fn in (("keyset", keyed), ("general", general)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[label].append(e0.elapsed_time(e1))
    st_k, st_g = d_st_k.cpu().numpy(), d_st_g.cpu().numpy()
    mism = int((st_k != st_g).sum())
    exp_mism = None if schnorr else int((st_g != expect).sum())
    ks.close()
    mk, mg = statistics.median(times["keyset"]), statistics.median(times["general"])
    return {
        "n": n, "keys": int(nkeys), "extra_invalid_keys": int(keys.shape[0] - nkeys), "schnorr": bool(schnorr),
        "keyset_ms": mk, "general_ms": mg, "speedup": mg / mk,
        "keyset_sigs_per_s": n / (mk * 1e-3), "general_sigs_per_s": n / (mg * 1e-3),
        "keyset_ms_all": times["keyset"], "general_ms_all": times["general"],
        "build_ms": build_ms, "table_bytes": int(keys.shape[0]) * 393216,
        "status_mismatches": mism, "general_vs_expected_mismatches": exp_mism,
        "statuses": {int(k): int(v) for k, v in zip(*np.unique(st_k, return_counts=True))},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--keys", type=str, default="1,1024,65536")
    ap.add_argument("--no-dkg", action="store_true")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if a.reps < 5:
        sys.exit("--reps must be at least 5")
    if not torch.cuda.is_available():
        sys.exit("bench_keyset: no CUDA device (there is no CPU path)")
    kb = importlib.import_module("kyber-rs_b200")
    ctx = kb.Context(0)
    n = 1 << LOG2N
    rng = np.random.default_rng(2024)
    res = {"metric": "key-set verify vs general verify, CUDA-event ms per 2^20 signatures (median)", **gpu_info(), "reps": a.reps, "configs": {}}
    for k in (int(x) for x in a.keys.split(",") if x):
        key_idx = rng.integers(0, k, size=n, dtype=np.uint32)
        res["configs"][f"K={k}"] = run_config(kb, ctx, f"K{k}", k, key_idx, False, a.reps)
        print(f"K={k}: {res['configs'][f'K={k}']['keyset_ms']:.3f} ms vs {res['configs'][f'K={k}']['general_ms']:.3f} ms", file=sys.stderr)
    if not a.no_dkg:
        key_idx = np.repeat(np.arange(1024, dtype=np.uint32), n // 1024)
        res["configs"]["dkg_1024x1024_schnorr"] = run_config(kb, ctx, "dkg", 1024, key_idx, True, a.reps)
    ok = all(c["status_mismatches"] == 0 and not c["general_vs_expected_mismatches"] for c in res["configs"].values())
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
