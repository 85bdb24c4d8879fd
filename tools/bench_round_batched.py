"""DKG rounds with KB_ROUND_CHECK_BATCHED against KB_ROUND_CHECK_EXACT on the same inputs.

Inputs: the round of tools/bench_dkg_keyed.py (cfg4: n = 1024 dealers and verifiers, t = 683; PriPoly::eval on the device;
2^20 deal and response signatures under 1024 participant keys), with the shares of 0, 1, 32, 341 or 1024 dealers
spoiled (one share each) for the share-check measurements and 0 or 1 (and the spoiling of tools/bench_dkg_keyed.py, which
reaches every dealer) for the keyed rounds, and cfg3 (n = 256, t = 171, honest shares plus one spoiled
dealer).  Timed, alternating the two modes on two contexts (median of --reps runs after one warm-up each):
  * share checks, device buffers, CUDA events on one stream: kb_dev_dkg_verify_round;
  * share checks, host buffers, host clock (the call ends in a synchronise): kb_dkg_verify_round;
  * the whole keyed round, device buffers: kb_dev_dkg_process_round_keyed;
  * the keyed round on every visible GPU, host buffers: kb_mctx_dkg_process_round_keyed.
Every verdict and status of every timed BATCHED run is compared item by item with the EXACT run before it, and the
fallback count with the number of spoiled dealers; any mismatch exits non-zero.  One JSON line on stdout (and in --out),
with the GPU's name, power limit and max SM clock read in the same run.  Also: the honest cfg4 round (all 1 024 dealers and
the 128 dealers of one GPU of eight) at every chunk count of k_rc_msm (KB_RC_CHUNKS), and its kernel times from one
torch.profiler run of their own.

  python tools/bench_round_batched.py [--reps 5] [--out profiles/r9_bench_round_batched.json]
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
from bench_dkg_keyed import cuda_ms, gpu_info, host_ms, signed_batch  # noqa: E402

FAIL = {"ok": True}


def check(cond, what):
    if not cond:
        FAIL["ok"] = False
        print("MISMATCH:", what, file=sys.stderr)


def spoil(shares, n, nd, nbad, tag):
    """one share of each of nbad dealers (spread over the round) changed"""
    out = shares.copy()
    dealers = np.unique(np.linspace(0, nd - 1, nbad).astype(np.int64)) if nbad else np.zeros(0, dtype=np.int64)
    assert dealers.size == nbad
    idx = dealers * n + (dealers * 37) % n
    out[idx, 4] ^= 0x40
    return out


def alternate_pair(run, reps, timer):
    """run(mode) -> outputs; timed alternately, every BATCHED output compared with the EXACT one before it"""
    times = {"exact": [], "batched": []}
    run("exact")
    run("batched")
    for _ in range(reps):
        want = None
        for mode in ("exact", "batched"):
            out = {}
            times[mode].append(timer(lambda: out.update(r=run(mode))))
            if mode == "exact":
                want = out["r"]
            else:
                got = out["r"]
                check(all((np.asarray(a) == np.asarray(b)).all() for a, b in zip(got, want)), "outputs")
    me, mb = statistics.median(times["exact"]), statistics.median(times["batched"])
    return {"exact_ms": me, "batched_ms": mb, "speedup": me / mb, "exact_ms_all": times["exact"], "batched_ms_all": times["batched"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_round_batched: no CUDA device (there is no CPU path)")
    kb = importlib.import_module("kyber-rs_b200")
    ngpu = torch.cuda.device_count()
    res = {"metric": "DKG round share checks and keyed rounds, KB_ROUND_CHECK_BATCHED vs EXACT, ms (median)", **gpu_info(), "reps": a.reps, "n_gpus_multi": ngpu}
    ctx = {"exact": kb.Context(0), "batched": kb.Context(0)}
    ctx["batched"].set_round_check("batched")
    c0 = ctx["exact"]
    dev = torch.device("cuda", 0)
    up = lambda x: torch.from_numpy(x.view(np.int64) if x.dtype == np.uint64 else np.ascontiguousarray(x)).to(dev)

    def share_checks(n, t, nbad_list, tag):
        coeffs = bench.xof(f"{tag}/coeffs", 32 * n * t).reshape(n * t, 32).copy()
        coeffs[:, 31] &= 0x0F
        commits = c0.point_mul_base_batch(coeffs, 1)
        honest = c0.pripoly_eval_batch(coeffs, t, n).copy()
        out = {}
        d_c = up(commits)
        for nbad in nbad_list:
            shares = spoil(honest, n, n, nbad, tag)
            d_s = up(shares)
            v = {m: torch.full((n * n,), 99, dtype=torch.uint8, device=dev) for m in ctx}

            def run_dev(mode):
                ctx[mode].dev_dkg_verify_round(n, t, n, d_c, d_s, v[mode])
                return None

            # timing on events only; the outputs of every timed pair are compared after it
            times = {"exact": [], "batched": []}
            for m in ctx:
                run_dev(m)
            for _ in range(a.reps):
                for m in ("exact", "batched"):
                    times[m].append(cuda_ms(lambda: run_dev(m)))
                check((v["exact"] == v["batched"]).all().item(), f"dev n={n} nbad={nbad}")
                check(ctx["batched"].round_fallbacks() == nbad, f"fallbacks n={n} nbad={nbad}")
            me, mb = statistics.median(times["exact"]), statistics.median(times["batched"])
            r = {"device_buffers": {"exact_ms": me, "batched_ms": mb, "speedup": me / mb, "exact_ms_all": times["exact"], "batched_ms_all": times["batched"]}}
            r["host_buffers"] = alternate_pair(lambda m: [ctx[m].dkg_verify_round(n, t, commits, shares)], a.reps, host_ms)
            check(ctx["batched"].round_fallbacks() == nbad, f"host fallbacks n={n} nbad={nbad}")
            r["verdict_zeros"] = int((v["exact"] == 0).sum().item())
            out[str(nbad)] = r
            del d_s, v
        return out

    res["cfg4_share_checks"] = {"n": 1024, "t": 683, "by_failing_dealers": share_checks(1024, 683, [0, 1, 32, 341, 1024], "kyber-b200/rc-cfg4")}
    res["cfg3_share_checks"] = {"n": 256, "t": 171, "by_failing_dealers": share_checks(256, 171, [0, 1], "kyber-b200/rc-cfg3")}
    torch.cuda.empty_cache()

    # ---- the chunk split of k_rc_msm (KB_RC_CHUNKS, read at context creation) on the honest cfg4 round: all 1 024 dealers,
    # and the 128 dealers one GPU of eight holds; plus the kernel times of each from a profiled run of its own
    n, t = 1024, 683
    tag = "kyber-b200/rc-cfg4"
    coeffs = bench.xof(f"{tag}/coeffs", 32 * n * t).reshape(n * t, 32).copy()
    coeffs[:, 31] &= 0x0F
    d_c = up(c0.point_mul_base_batch(coeffs, 1))
    d_s = up(c0.pripoly_eval_batch(coeffs, t, n).copy())
    want = {}
    for nd in (n, 128):
        vx = torch.empty(nd * n, dtype=torch.uint8, device=dev)
        c0.dev_dkg_verify_round(n, t, nd, d_c, d_s, vx)
        want[nd] = vx
    sweep = {}
    for chunks in (0, 1, 2, 4, 5, 8, 16):
        if chunks:
            os.environ["KB_RC_CHUNKS"] = str(chunks)
        cc = kb.Context(0)
        os.environ.pop("KB_RC_CHUNKS", None)
        cc.set_round_check("batched")
        row = {}
        for nd in (n, 128):
            vb = torch.empty(nd * n, dtype=torch.uint8, device=dev)
            run = lambda: cc.dev_dkg_verify_round(n, t, nd, d_c, d_s, vb)
            run()
            row[str(nd)] = statistics.median(cuda_ms(run) for _ in range(a.reps))
            check((vb == want[nd]).all().item() and cc.round_fallbacks() == 0, f"chunks={chunks} nd={nd}")
        sweep["default" if chunks == 0 else str(chunks)] = row
        cc.close()
    res["cfg4_honest_batched_ms_by_chunks"] = sweep
    prof_ms = {}
    for nd in (n, 128):
        vb = torch.empty(nd * n, dtype=torch.uint8, device=dev)
        ctx["batched"].dev_dkg_verify_round(n, t, nd, d_c, d_s, vb)
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ctx["batched"].dev_dkg_verify_round(n, t, nd, d_c, d_s, vb)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            if us:
                kern[ev.key[:60]] = round(us / 3 / 1e3, 4)
        prof_ms[str(nd)] = dict(sorted(kern.items(), key=lambda kv: -kv[1]))
    res["cfg4_honest_batched_kernel_ms_per_call_by_dealers"] = prof_ms
    del d_c, d_s, want
    torch.cuda.empty_cache()

    # ---- the whole keyed round (the inputs of tools/bench_dkg_keyed.py)
    n, t = 1024, 683
    m = n * n
    tag = "kyber-b200/dkg-keyed"
    coeffs = bench.xof(f"{tag}/coeffs", 32 * n * t).reshape(n * t, 32).copy()
    coeffs[:, 31] &= 0x0F
    commits = c0.point_mul_base_batch(coeffs, 1)
    honest = c0.pripoly_eval_batch(coeffs, t, n).copy()
    inputs = {"honest": (honest, 0), "one_dealer_spoiled": (spoil(honest, n, n, 1, tag), 1)}
    every = honest.copy()
    every[::251, 3] ^= 0x10   # the inputs of tools/bench_dkg_keyed.py: every dealer has a wrong share
    inputs["every_251st_share_spoiled"] = (every, len({k // n for k in range(0, m, 251)}))
    seeds = bench.xof(f"{tag}/seeds", 32 * n).reshape(n, 32).copy()
    k = np.arange(m)
    deal = signed_batch(c0, seeds, k // n, 128, f"{tag}/deal")
    resp = signed_batch(c0, seeds, k % n, 32, f"{tag}/resp")
    keys = deal[3][::n].copy()
    ks = {mo: ctx[mo].keyset(keys) for mo in ctx}
    d_c = up(commits)
    d_deal, d_resp = [up(x) for x in deal[:3]], [up(x) for x in resp[:3]]
    outs = {mo: [torch.full((m,), 99, dtype=torch.uint8, device=dev) for _ in range(3)] for mo in ctx}
    res["cfg4_keyed_round_device_buffers"] = {}
    for name, (shares, spoiled) in inputs.items():
        d_s = up(shares)

        def keyed(mode):
            v, ds, rs = outs[mode]
            ctx[mode].dev_dkg_process_round_keyed(n, t, n, d_c, d_s, v, ks[mode], deal=(*d_deal, ds), resp=(*d_resp, rs))

        times = {"exact": [], "batched": []}
        for mo in ctx:
            keyed(mo)
        for _ in range(a.reps):
            for mo in ("exact", "batched"):
                times[mo].append(cuda_ms(lambda: keyed(mo)))
            check(all((x == y).all().item() for x, y in zip(outs["exact"], outs["batched"])), f"keyed round {name}")
            check(ctx["batched"].round_fallbacks() == spoiled, f"keyed fallbacks {name}")
        me, mb = statistics.median(times["exact"]), statistics.median(times["batched"])
        res["cfg4_keyed_round_device_buffers"][name] = {"spoiled_dealers": spoiled, "exact_ms": me, "batched_ms": mb, "speedup": me / mb, "exact_ms_all": times["exact"], "batched_ms_all": times["batched"]}
        del d_s

    for mo in ctx:
        ks[mo].close()
        ctx[mo].close()
    del d_c, d_deal, d_resp, outs
    torch.cuda.empty_cache()

    # ---- the keyed round on every visible GPU, host buffers
    mctx = {mo: kb.MultiContext(list(range(ngpu))) for mo in ("exact", "batched")}
    mctx["batched"].set_round_check("batched")
    mk = {mo: mctx[mo].keyset(keys) for mo in mctx}
    res["cfg4_keyed_round_multi_gpu_host_buffers"] = {}
    for name in ("honest", "one_dealer_spoiled"):
        shares = inputs[name][0]
        r = alternate_pair(lambda mo: list(mctx[mo].dkg_process_round_keyed(n, t, commits, shares, mk[mo], deal=deal[:3], resp=resp[:3])), a.reps, host_ms)
        res["cfg4_keyed_round_multi_gpu_host_buffers"][name] = r
    for mo in mctx:
        mk[mo].close()
        mctx[mo].close()
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
