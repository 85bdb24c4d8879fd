"""A/B of two builds of libkyber_b200.so on the headline verify workload, in one process tree on one GPU.

    python tools/ab_verify_wrap.py --base build/ab/base.so --new kyber-rs_b200/libkyber_b200.so --runs 5 --out /tmp/ab

Runs `bench.py --no-extras --steps K` alternately with each library (KYBER_B200_LIB), `runs` times each, the order of the two
swapped every pair; then `--dump-outputs` once per build and compares the dumps.  Prints one line per run, the medians, the
per-pair ratios and the spread of each build, and writes the raw bench lines, the card's name, power limit and clock, and
the summary under --out.  Used for the short-wrap field bodies of the main verify kernel (profiles/r6_ab_short_wrap*.txt)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(lib, steps, dump=None):
    env = dict(os.environ, KYBER_B200_LIB=os.path.abspath(lib))
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--no-extras", "--steps", str(steps)]
    if dump:
        cmd += ["--dump-outputs", dump]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=ROOT)
    if r.returncode != 0:
        raise RuntimeError(f"bench.py with {lib} failed ({r.returncode}):\n{r.stderr[-3000:]}")
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    return line, json.loads(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True)
    ap.add_argument("--new", required=True)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    log = open(os.path.join(a.out, "ab.txt"), "w")

    def say(s):
        print(s, flush=True)
        log.write(s + "\n")

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    say(f"# card: {smi}")
    say(f"# bench.py --no-extras --steps {a.steps}, {a.runs} runs per build, alternating")
    libs = {"base": a.base, "new": a.new}
    res = {"base": [], "new": []}
    raw = open(os.path.join(a.out, "bench_lines.jsonl"), "w")
    for r in range(a.runs):
        order = ("base", "new") if r % 2 == 0 else ("new", "base")
        for tag in order:
            line, d = bench(libs[tag], a.steps)
            raw.write(json.dumps({"build": tag, "run": r, "bench": d}) + "\n")
            km = d["roofline"]["kernels_ms"]
            res[tag].append((d["value"], km["k_verify_half_prep"], km["k_verify_half_main"]))
            say(f"run {r} {tag:4s} value {d['value']:.4g} {d.get('unit', '')}  prep {km['k_verify_half_prep']:.3f} ms  main {km['k_verify_half_main']:.3f} ms")
    for tag in ("base", "new"):
        v = [x[0] for x in res[tag]]
        say(f"{tag}: median value {statistics.median(v):.4g} (min {min(v):.4g} max {max(v):.4g}, spread {100 * (max(v) - min(v)) / statistics.median(v):.2f} %), "
            f"median prep {statistics.median(x[1] for x in res[tag]):.3f} ms, median main {statistics.median(x[2] for x in res[tag]):.3f} ms")
    ratios = [n[0] / b[0] for b, n in zip(res["base"], res["new"])]
    say("pair ratios new/base: " + " ".join(f"{x:.4f}" for x in ratios) + f"  median {statistics.median(ratios):.4f}")
    dumps = {}
    for tag in ("base", "new"):
        d = os.path.join(a.out, f"dump_{tag}")
        bench(libs[tag], 2, dump=d)
        dumps[tag] = {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith(".npy")}
    same = dumps["base"].keys() == dumps["new"].keys() and all(np.array_equal(dumps["base"][k], dumps["new"][k]) for k in dumps["base"])
    say(f"dump-outputs identical: {same} ({', '.join(f'{k} {v.shape}' for k, v in dumps['new'].items())})")
    log.close()
    return 0 if same else 1


if __name__ == "__main__":
    sys.exit(main())
