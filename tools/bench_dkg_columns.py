"""The share checks of a DKG round for a range of k verifiers (kb_dkg_verify_columns) against today's per-share route.

Inputs: cfg4 (n = 1 024 dealers and verifiers, t = 683; commitments and PriPoly::eval on the device), one share in every
97th spoiled.  For k = 1, 4, 6, 8, 16, 64 and 256 columns from ver_lo = 333, timed alternately (median of --reps runs after one
warm-up each):
  * kb_dev_dkg_verify_columns in EXACT and BATCHED mode (device buffers, CUDA events on one stream), and with each route
    forced (KB_DKG_COLUMNS=1: the column kernel, =0: the per-share Horner kernel on the items), for the planner's crossover;
  * kb_dkg_verify_columns in EXACT and BATCHED mode from host buffers (host clock; the call ends in a synchronise);
  * kb_vss_verify_deals_batch on the same items (poly_id = d, idx = i), host buffers: the only route before this call;
  * the whole round (kb_dev_dkg_verify_round, EXACT and BATCHED) times k / n, the share of a round these columns are.
Every verdict array of every timed run is compared item by item with the kb_vss_verify_deals_batch run, which is checked
first; any mismatch exits non-zero.  Kernel times of the column route at k = 1 and 64 come from one torch.profiler run of
their own.  One JSON line on stdout (and in --out), with the GPU's name, power limit and max SM clock read in the same run.

  python tools/bench_dkg_columns.py [--reps 7] [--out profiles/r10_bench_dkg_columns.json]
"""
import argparse
import importlib
import json
import os
import statistics
import sys

import numpy as np
import torch

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_dkg_keyed import cuda_ms, gpu_info, host_ms  # noqa: E402

FAIL = {"ok": True}
KS = (1, 4, 6, 8, 16, 64, 256)
VER_LO = 333


def check(cond, what):
    if not cond:
        FAIL["ok"] = False
        print("MISMATCH:", what, file=sys.stderr)


def context(kb, mode, columns=None):
    if columns is not None:
        os.environ["KB_DKG_COLUMNS"] = columns
    try:
        c = kb.Context(0)
    finally:
        os.environ.pop("KB_DKG_COLUMNS", None)
    c.set_round_check(mode)
    return c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    kb = importlib.import_module("kyber-rs_b200")
    res = {"bench": "dkg_columns", **gpu_info(), "n": 1024, "t": 683, "dealers": 1024, "ver_lo": VER_LO, "reps": a.reps}
    ctx = {"exact": context(kb, "exact"), "batched": context(kb, "batched"), "column_route": context(kb, "exact", "1"), "per_share_route": context(kb, "exact", "0")}
    c0 = ctx["exact"]
    n, t = 1024, 683
    tag = "kyber-b200/dkg-columns"
    coeffs = bench.xof(f"{tag}/coeffs", 32 * n * t).reshape(n * t, 32).copy()
    coeffs[:, 31] &= 0x0F
    commits = c0.point_mul_base_batch(coeffs, 1).copy()
    shares = c0.pripoly_eval_batch(coeffs, t, n).copy()
    shares[::97, 4] ^= 0x40
    dev = torch.device("cuda", 0)

    def up(x):
        return torch.from_numpy(np.ascontiguousarray(x)).to(dev)

    d_c = up(commits)
    d_full = up(shares)
    v_full = {mo: torch.zeros(n * n, dtype=torch.uint8, device=dev) for mo in ("exact", "batched")}
    for mo in v_full:
        ctx[mo].dev_dkg_verify_round(n, t, n, d_c, d_full, v_full[mo])
    round_ms = {"exact": [], "batched": []}
    for _ in range(a.reps):
        for mo in round_ms:
            round_ms[mo].append(cuda_ms(lambda: ctx[mo].dev_dkg_verify_round(n, t, n, d_c, d_full, v_full[mo])))
    check((v_full["exact"] == v_full["batched"]).all().item(), "full round exact vs batched")
    res["full_round_device_ms"] = {mo: statistics.median(v) for mo, v in round_ms.items()}
    del d_full
    res["columns"] = {}
    for k in KS:
        lo, hi = VER_LO, VER_LO + k
        sh = shares.reshape(n, n, 32)[:, lo:hi].reshape(-1, 32).copy()
        pid = np.repeat(np.arange(n, dtype=np.uint32), k)
        idx = np.tile(np.arange(lo, hi, dtype=np.uint32), n)
        want = c0.vss_verify_deals_batch(commits, t, pid, idx, sh)
        check(want.any() and not want.all(), f"k={k}: the reference has both verdicts")
        for name, c in ctx.items():
            check((c.dkg_verify_columns(n, t, commits, sh, lo, hi) == want).all(), f"k={k} host {name}")
        d_s = up(sh)
        d_v = {name: torch.full((n * k,), 7, dtype=torch.uint8, device=dev) for name in ctx}
        times = {name: [] for name in ctx}
        times.update({f"host_{mo}": [] for mo in ("exact", "batched")})
        times["vss_verify_deals_batch_host"] = []
        for name in ctx:
            ctx[name].dev_dkg_verify_columns(n, t, n, d_c, d_s, d_v[name], lo, hi)
        c0.vss_verify_deals_batch(commits, t, pid, idx, sh)
        for _ in range(a.reps):
            for name in ctx:
                times[name].append(cuda_ms(lambda: ctx[name].dev_dkg_verify_columns(n, t, n, d_c, d_s, d_v[name], lo, hi)))
                check((d_v[name].cpu().numpy() == want).all(), f"k={k} device {name}")
            for mo in ("exact", "batched"):
                out = {}
                times[f"host_{mo}"].append(host_ms(lambda: out.setdefault("v", ctx[mo].dkg_verify_columns(n, t, commits, sh, lo, hi))))
                check((out["v"] == want).all(), f"k={k} host {mo}")
            out = {}
            times["vss_verify_deals_batch_host"].append(host_ms(lambda: out.setdefault("v", c0.vss_verify_deals_batch(commits, t, pid, idx, sh))))
            check((out["v"] == want).all(), f"k={k} vss_verify_deals_batch")
        r = {f"{name}_ms": statistics.median(v) for name, v in times.items()}
        r["full_round_share_ms"] = {mo: v * k / n for mo, v in res["full_round_device_ms"].items()}
        r["speedup_vs_vss_verify_deals_batch_host"] = r["vss_verify_deals_batch_host_ms"] / r["host_exact_ms"]
        r["all_ms"] = times
        res["columns"][str(k)] = r
        del d_s, d_v
    # kernel times of the column route, one profiler run of their own
    prof_out = {}
    for k in (1, 64):
        lo, hi = VER_LO, VER_LO + k
        d_s = up(shares.reshape(n, n, 32)[:, lo:hi].reshape(-1, 32))
        d_v = torch.zeros(n * k, dtype=torch.uint8, device=dev)
        ctx["column_route"].dev_dkg_verify_columns(n, t, n, d_c, d_s, d_v, lo, hi)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as p:
            for _ in range(3):
                ctx["column_route"].dev_dkg_verify_columns(n, t, n, d_c, d_s, d_v, lo, hi)
            torch.cuda.synchronize()
        kt = {}
        for ev in p.key_averages():
            if ev.device_type == torch.autograd.DeviceType.CUDA or getattr(ev, "device_time_total", 0) > 0:
                us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                if us > 0:
                    kt[ev.key] = {"ms_per_call": us / 3 / 1e3, "launches_per_call": ev.count / 3}
        prof_out[str(k)] = kt
    res["column_route_kernel_times"] = prof_out
    for c in ctx.values():
        c.close()
    res["all_outputs_equal"] = FAIL["ok"]
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    sys.exit(0 if FAIL["ok"] else 1)


if __name__ == "__main__":
    main()
