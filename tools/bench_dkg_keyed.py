"""The whole DKG round (cfg4: n = 1024 dealers and verifiers, t = 683) with the deal and response signatures verified under
registered participant keys, against the same round with one pk per item, on the same inputs.

Inputs: every dealer's polynomial and its 1024 shares (PriPoly::eval on the device, 0.4 % corrupted); 2^20 deal messages
of 128 bytes, deal k signed by participant k / n, and 2^20 responses of 32 bytes, response k signed by participant k % n,
every 8th signature damaged in s, R or the message.  1024 participant keys serve as both dealers and verifiers.

Timed, alternating the two calls (median of --reps runs after one warm-up each):
  * one GPU, device buffers, CUDA events on one stream: kb_dev_dkg_process_round_keyed against kb_dev_dkg_process_round;
  * all visible GPUs, host buffers, host clock around the calls (which end in a synchronise):
    kb_mctx_dkg_process_round_keyed against kb_mctx_dkg_process_round;
  * the key-set builds (kb_keyset_create, kb_mctx_keyset_create), host clock (both wait for the build).
Every verdict and status of the keyed calls is compared item by item with the unkeyed ones; any mismatch exits non-zero.
One JSON line on stdout (and in --out), with the GPU's name, power limit and max SM clock read in the same run.

  python tools/bench_dkg_keyed.py [--reps 7] [--out profiles/r4_bench_dkg_keyed.json]
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


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # pragma: no cover
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": None, "max_sm_clock": None, "nvidia_smi": str(e)}


def signed_batch(ctx, seeds, signer, mlen, tag):
    """(flat, off, sig): message k of mlen bytes signed by seeds[signer[k]]; every 8th item damaged in s, R or the message"""
    m = signer.shape[0]
    flat = bench.xof(f"{tag}/msgs", mlen * m).copy()
    off = np.arange(m + 1, dtype=np.uint64) * np.uint64(mlen)
    sig, pk = ctx.eddsa_sign_batch(seeds[signer], flat, off)
    sig = sig.copy()
    k = np.arange(3, m, 8)
    kind = (k // 8) % 3
    sig[k[kind == 0], 40] ^= 0x04
    sig[k[kind == 1], 5] ^= 0x20
    flat[mlen * k[kind == 2] + 7] ^= 1
    return flat, off, sig, pk.copy()


def make_round(ctx, n, t):
    tag = "kyber-b200/dkg-keyed"
    coeffs = bench.xof(f"{tag}/coeffs", 32 * n * t).reshape(n * t, 32).copy()
    coeffs[:, 31] &= 0x0F
    commits = ctx.point_mul_base_batch(coeffs, 1)
    shares = ctx.pripoly_eval_batch(coeffs, t, n).copy()
    shares[::251, 3] ^= 0x10
    seeds = bench.xof(f"{tag}/seeds", 32 * n).reshape(n, 32).copy()
    k = np.arange(n * n)
    deal = signed_batch(ctx, seeds, k // n, 128, f"{tag}/deal")
    resp = signed_batch(ctx, seeds, k % n, 32, f"{tag}/resp")
    keys = deal[3][::n].copy()          # the key of dealer d signed deal d * n
    assert (keys[k % n] == resp[3]).all()
    return commits, shares, deal, resp, keys


def alternate(fns, reps, timer):
    for fn in fns.values():
        fn()
    times = {label: [] for label in fns}
    for _ in range(reps):
        for label, fn in fns.items():
            times[label].append(timer(fn))
    return times


def cuda_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def host_ms(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def summary(times, keyed, general):
    mk, mg = statistics.median(times[keyed]), statistics.median(times[general])
    return {"keyed_ms": mk, "general_ms": mg, "speedup": mg / mk, "keyed_ms_all": times[keyed], "general_ms_all": times[general]}


def mismatches(a, b):
    return sum(int((x != y).sum()) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024)
    ap.add_argument("--t", type=int, default=683)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if a.reps < 5:
        sys.exit("--reps must be at least 5")
    if not torch.cuda.is_available():
        sys.exit("bench_dkg_keyed: no CUDA device (there is no CPU path)")
    kb = importlib.import_module("kyber-rs_b200")
    n, t = a.n, a.t
    m = n * n
    ngpu = torch.cuda.device_count()
    res = {"metric": "DKG round (share checks + 2 x n^2 Schnorr verifies) under registered participant keys vs one pk per item, ms (median)",
           **gpu_info(), "n": n, "t": t, "deal_msg_bytes": 128, "resp_msg_bytes": 32, "reps": a.reps, "n_gpus_multi": ngpu}
    ctx = kb.Context(0)
    t0 = time.perf_counter()
    commits, shares, deal, resp, keys = make_round(ctx, n, t)
    res["prep_s"] = time.perf_counter() - t0
    k = np.arange(m)

    # ---- one GPU, device buffers
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ks = ctx.keyset(keys)
    res["keyset_build_ms"] = (time.perf_counter() - t0) * 1e3
    res["keyset_bytes_per_gpu"] = n * 393216
    dev = torch.device("cuda", 0)
    up = lambda x: torch.from_numpy(x.view(np.int64) if x.dtype == np.uint64 else np.ascontiguousarray(x)).to(dev)
    d_c, d_s = up(commits), up(shares)
    d_deal, d_resp = [up(x) for x in deal[:3]], [up(x) for x in resp[:3]]
    d_dpk, d_rpk = up(keys[k // n]), up(keys[k % n])
    outs = {lbl: [torch.full((m,), 99, dtype=torch.uint8, device=dev) for _ in range(3)] for lbl in ("keyed", "general")}

    def dev_keyed():
        v, ds, rs = outs["keyed"]
        ctx.dev_dkg_process_round_keyed(n, t, n, d_c, d_s, v, ks, deal=(*d_deal, ds), resp=(*d_resp, rs))

    def dev_general():
        v, ds, rs = outs["general"]
        ctx.dev_dkg_process_round(n, t, n, d_c, d_s, v, deal=(d_dpk, *d_deal, ds), resp=(d_rpk, *d_resp, rs))

    times = alternate({"keyed": dev_keyed, "general": dev_general}, a.reps, cuda_ms)
    res["one_gpu_device_buffers"] = summary(times, "keyed", "general")
    got = [x.cpu().numpy() for x in outs["keyed"]]
    want = [x.cpu().numpy() for x in outs["general"]]
    res["one_gpu_mismatches"] = mismatches(got, want)
    res["statuses"] = {name: {int(s): int(c) for s, c in zip(*np.unique(x, return_counts=True))} for name, x in zip(("verdict", "deal", "resp"), want)}
    del d_c, d_s, d_deal, d_resp, d_dpk, d_rpk, outs
    ks.close()
    ctx.close()
    torch.cuda.empty_cache()

    # ---- all visible GPUs, host buffers
    mctx = kb.MultiContext(list(range(ngpu)))
    t0 = time.perf_counter()
    mk = mctx.keyset(keys)
    res["multi_keyset_build_ms"] = (time.perf_counter() - t0) * 1e3
    host = {lbl: [np.full(m, 99, dtype=np.uint8) for _ in range(3)] for lbl in ("keyed", "general")}
    dpk, rpk = keys[k // n], keys[k % n]

    def multi_keyed():
        v, ds, rs = mctx.dkg_process_round_keyed(n, t, commits, shares, mk, deal=deal[:3], resp=resp[:3], verdict=host["keyed"][0])
        host["keyed"][1:] = [ds, rs]

    def multi_general():
        v, ds, rs = mctx.dkg_process_round(n, t, commits, shares, deal=(dpk, *deal[:3]), resp=(rpk, *resp[:3]), verdict=host["general"][0])
        host["general"][1:] = [ds, rs]

    times = alternate({"keyed": multi_keyed, "general": multi_general}, a.reps, host_ms)
    res["multi_gpu_host_buffers"] = summary(times, "keyed", "general")
    res["multi_gpu_mismatches"] = mismatches(host["keyed"], host["general"])
    res["one_vs_multi_mismatches"] = mismatches(host["keyed"], got)
    mk.close()
    mctx.close()
    ok = res["one_gpu_mismatches"] == 0 and res["multi_gpu_mismatches"] == 0 and res["one_vs_multi_mismatches"] == 0
    res["all_outputs_equal"] = ok
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
