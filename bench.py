#!/usr/bin/env python
"""bench.py — benchmark of the edwards25519 hot path (BASELINE.json metric), with parity checks in the code path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--log2n 20] [--no-extras] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes, on rank 0, what the last timed step returned: the statuses of the device-resident verify
(verify_status.npy) and of the host-buffer verify (e2e_verify_status.npy), as float32.  The inputs depend only on the
arguments, so two builds can be compared output for output.

Headline (config.workload): BASELINE.json configs[1] — batched EdDSA verification
(eddsa::verify_with_checks, sign/eddsa/eddsa_sig.rs:159-212) of 2^20 random keys / 64-byte messages / signatures
per GPU, including the per-signature SHA-512 challenge; 1/64 of the items are deliberately invalid (nine classes).
A "step" is one pass over that batch.  One process per GPU; every rank owns its own 2^20 signatures (weak scaling,
independent shards, no data-path collective).

  value         verified signatures / s, inputs resident in HBM (CUDA events on the launch stream), all ranks
  e2e           the same metric from HOST buffers through the C ABI's multi-device context (kb_mctx_verify_batch):
                rank 0 hands ONE batch of N x 2^20 signatures to all N GPUs (H2D + D2H inside the timed region)
  roofline      integer-multiply roofline of the verify step, 154 k IMAD-eq CHARGED per signature (SURVEY 8d), against
                the ARCHITECTURAL IMAD.WIDE rate 32 lanes x SMs x clock (kb_probe_imad's streams are reported next to it)
  cpu_baseline  the oracle's ref10-style C port (oracle/ref10_port.c) on the host cores, on a prefix of the same batch
  configs       BASELINE configs 1, 3, 4, 5 as first-class entries: value, roofline, e2e, cpu_baseline (N = 1), with the
                STRONG-scaling shapes (cfg4: the fixed n = 1024 round split by dealer; cfg5: 2^16..2^26 TOTAL points)
  stages        the pure decompress and hash stages: achieved HBM GB/s
  parity_checked what was compared with the oracle / with expected verdicts inside this very run (any mismatch exits non-zero)

--impl reference times the CPU port on all host cores on a prefix of the SAME batch (the reference is Rust; there is no
Rust toolchain in this image, see DESIGN.md).
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True     # the benchmark writes nothing into the source tree, which may be read-only
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# ---- algorithmic work per unit, SURVEY §8(d): M = 72, S = 44 IMAD-eq -------------------------------------------------
IMAD_EQ_PER_VERIFY = 154_000      # A decompress + Straus s*B - h*A + compress (the CHARGED figure)
IMAD_EQ_PER_BASE_MUL = 32_500
IMAD_EQ_PER_VAR_MUL = 138_300
IMAD_EQ_PER_EVAL_COEFF = 6_800    # PubPoly::eval per coefficient (x <= 1024)
IMAD_EQ_PER_MSM_POINT = 20_700
IMAD_EQ_PER_DECOMPRESS = 20 * 72 + 255 * 44
# what the half-size-scalar kernels execute per signature (IMAD.WIDE, M = 73, S = 44; DESIGN.md §3.6):
EXEC_PREP_PER_VERIFY = 25_600
EXEC_MAIN_PER_VERIFY = 101_200   # 127.3 doublings x 413 + 63.6 joint-table additions x 555 (records sorted by length; the first operand is taken as it is) + 15 comb additions x 482 (affine operands) + 6.1 k for the joint table
ALG_BYTES_PER_SIG = 161           # 32 pk + 64 sig + 64 msg + 1 status
L_ORDER = 2**252 + 27742317777372353535851937790883648493
WEAK_R = bytes.fromhex("c7176a703d4dd84fba3c0b760d10670f2a2053fa2c39ccc64ec7fd7792ac037a")
NONCANON = bytes([0xEF]) + b"\xff" * 31
T8 = bytes.fromhex("26e8958fc2b227b045c3f489f2ef98f0d5dfac05d3c63339b13802886d53fc05")   # a point of order 8
OFF_CURVE = bytes.fromhex("02" + "00" * 31)     # y = 2: (y^2 - 1) / (d y^2 + 1) is not a square (checked against the oracle below)
INVALID_CLASSES = 9


def a1_range(i: int) -> bytes:
    """A canonical y that Point::is_canonical reports non-canonical (SURVEY §A1): low byte in [0x14, 0xEC]."""
    return bytes([0x14 + (i % 0xD9)]) + b"\xff" * 30 + b"\x7f"


def xof(seed: str, n: int) -> np.ndarray:
    import blake3

    return np.frombuffer(blake3.blake3(seed.encode()).digest(length=n), dtype=np.uint8)


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        return os.cpu_count() or 1


# ---- the cfg2 batch: identical items for both arms --------------------------------------------------------------------
def batch_secrets(n: int, rank: int):
    """Keys, nonces and messages of batch `rank` (BLAKE3-XOF of an ASCII seed, the reference's suite.xof construction)."""
    tag = f"kyber-b200/cfg2/rank{rank}"
    a = xof(tag + "/keys", 32 * n).reshape(n, 32).copy()
    a[:, 0] &= 0xF8
    a[:, 31] &= 0x7F
    a[:, 31] |= 0x40                        # curve.rs:79-84 clamp: unreduced scalar, bit 254 set
    r = xof(tag + "/nonces", 32 * n).reshape(n, 32).copy()
    r[:, 31] &= 0x0F                        # < 2^252 < L
    msg = xof(tag + "/msgs", 64 * n).copy()
    return a, r, msg


def spoil(pk, msg, sig, lo: int, hi: int):
    """Every 64th item of [lo, hi) is made invalid, cycling through nine classes; returns the statuses expected by
    construction (the reference's check order, eddsa_sig.rs:159-212)."""
    expect = np.zeros(hi - lo, dtype=np.uint8)
    for i in range(lo + ((63 - lo) % 64), hi, 64):
        k, j = (i // 64) % INVALID_CLASSES, i - lo
        if k == 0:
            msg[64 * j] ^= 1; expect[j] = 8                                  # flipped message bit -> InvalidSignature
        elif k == 1:
            v = (int.from_bytes(sig[j, 32:].tobytes(), "little") + L_ORDER) % (1 << 256)
            sig[j, 32:] = np.frombuffer(v.to_bytes(32, "little"), dtype=np.uint8); expect[j] = 2   # s + L
        elif k == 2:
            sig[j, :32] = np.frombuffer(NONCANON, dtype=np.uint8); expect[j] = 3
        elif k == 3:
            sig[j, :32] = np.frombuffer(WEAK_R, dtype=np.uint8); expect[j] = 4
        elif k == 4:
            pk[j] = np.frombuffer(WEAK_R, dtype=np.uint8); expect[j] = 6
        elif k == 5:
            pk[j] = np.frombuffer(NONCANON, dtype=np.uint8); expect[j] = 5
        elif k == 6:
            sig[j, :32] = np.frombuffer(OFF_CURVE, dtype=np.uint8); expect[j] = 7      # R is not a curve point -> MarshallingError
        elif k == 7:
            sig[j, :32] = np.frombuffer(a1_range(i), dtype=np.uint8); expect[j] = 3    # §A1 quirk range in R
        else:
            pk[j] = np.frombuffer(a1_range(i), dtype=np.uint8); expect[j] = 5          # §A1 quirk range in the key
    return expect


def make_batch(ctx, n: int, rank: int):
    """Synthetic signatures, signed WITH the library's own batched primitives (fixed-base mul, challenge hash,
    sc_mul_add — the signing equations of schnorr_sig.rs:25-47); spot-checked against the oracle by the caller."""
    a, r, msg = batch_secrets(n, rank)
    off = (np.arange(n + 1, dtype=np.uint64) * np.uint64(64))
    pk = ctx.point_mul_base_batch(a)
    R = ctx.point_mul_base_batch(r)
    h = ctx.challenge_batch(R, pk, msg, off)
    s = ctx.sc_muladd_batch(h, a, r)
    sig = np.concatenate([R, s], axis=1)
    expect = spoil(pk, msg, sig, 0, n)
    return pk, msg, off, sig, expect


def make_batch_cpu(C, m: int, rank: int, n_full: int, threads: int):
    """The first m items of the SAME batch, signed with the oracle (no GPU involved): what the reference arm verifies."""
    a, r, msg = batch_secrets(n_full, rank)
    a, r, msg = a[:m], r[:m], msg[:64 * m].copy()
    off = (np.arange(m + 1, dtype=np.uint64) * np.uint64(64))
    pk = C.mul_base_batch(a, nthreads=threads)
    R = C.mul_base_batch(r, nthreads=threads)
    sig = np.empty((m, 64), dtype=np.uint8)
    sig[:, :32] = R
    for i in range(m):
        h = C.sc_reduce64(C.sha512(R[i].tobytes() + pk[i].tobytes() + msg[64 * i:64 * i + 64].tobytes()))
        sig[i, 32:] = np.frombuffer(C.sc_muladd(h, a[i].tobytes(), r[i].tobytes()), dtype=np.uint8)
    expect = spoil(pk, msg, sig, 0, m)
    return pk, msg, off, sig, expect


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.idx)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:  # pragma: no cover
            self.p.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def die(msg: str):
    sys.stderr.write("bench: PARITY FAILURE: " + msg + "\n")
    sys.stderr.flush()
    os._exit(3)     # non-zero for the driver; os._exit so that no other rank's barrier can hang the exit


DUMP_BYTES = 60 << 20     # all files of --dump-outputs together, .npy headers included, stay under 64 MB


def dump_outputs(out_dir: str, arrays: dict):
    """Writes every array as out_dir/<name>.npy in float32.  An array larger than its equal share of DUMP_BYTES is cut
    to a fixed sample: the elements at sorted indices drawn with seed 0 (the same for every run of the same size),
    whose indices go to <name>_index.npy as float64."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a).reshape(-1)
        if 4 * a.size > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share // 12, replace=False))
            np.save(os.path.join(out_dir, name + "_index.npy"), idx.astype(np.float64))
            a = a[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def cpu_verify_baseline(C, pk, msg, off, sig, gpu_status, budget_s: float, threads: int):
    """Times the oracle's C port on a bounded prefix (adaptive: ~budget_s of CPU work) and checks the GPU statuses of
    that prefix against it."""
    probe = 256
    t0 = time.perf_counter()
    C.verify_batch(pk[:probe], msg[: 64 * probe], off[: probe + 1], sig[:probe], nthreads=threads)
    rate = probe / (time.perf_counter() - t0)
    m = int(min(pk.shape[0], max(probe, rate * budget_s)))
    m -= m % 64
    t0 = time.perf_counter()
    st = C.verify_batch(pk[:m], msg[: 64 * m], off[: m + 1], sig[:m], nthreads=threads)
    dt = time.perf_counter() - t0
    if gpu_status is not None and not (st == gpu_status[:m]).all():
        die("GPU statuses differ from the oracle on the CPU-baseline prefix")
    sodium = None
    try:  # independent sanity anchor (SURVEY 8d): libsodium's own verifier, one core, same signatures
        import nacl.bindings as nb

        k = 0
        t1 = time.perf_counter()
        for i in range(min(m, 4000)):
            if gpu_status is not None and gpu_status[i] != 0:
                continue
            nb.crypto_sign_open(sig[i].tobytes() + msg[64 * i:64 * i + 64].tobytes(), pk[i].tobytes())
            k += 1
        sodium = k / (time.perf_counter() - t1)
    except Exception:  # pragma: no cover - optional
        pass
    return {"value": m / dt, "unit": "sigs/s", "cores": threads, "kind": "port", "libsodium_single_core_sigs_per_s": sodium,
            "libsodium_all_cores_equivalent_sigs_per_s": sodium * threads if sodium else None,
            "sample": f"first {m} of the 2^20 signatures of the same batch, oracle/ref10_port.c (ref10-style C restatement of the Rust path; no Rust toolchain in this image), {dt:.1f} s",
            "checked_items": m}


def run_reference(args, rank, world):
    """The reference arm: the CPU port of the reference's algorithm on all host cores, on a prefix of the SAME batch
    the GPU arm verifies (same seeds, same invalid mix), each step a bounded sample."""
    if rank != 0:
        return
    from helpers import load_c_oracle

    C = load_c_oracle()
    threads = host_cores()
    n_full = 1 << args.log2n
    NREF = min(n_full, 16384)
    pk, msg, off, sg, expect = make_batch_cpu(C, NREF, 0, n_full, threads)
    t0 = time.perf_counter()
    C.verify_batch(pk[:256], msg[: 64 * 256], off[:257], sg[:256], nthreads=threads)
    rate = 256 / (time.perf_counter() - t0)
    per_step = int(min(NREF, max(256, rate * 4.0)))
    per_step -= per_step % 64
    for _ in range(args.warmup):
        C.verify_batch(pk[:per_step], msg[: 64 * per_step], off[: per_step + 1], sg[:per_step], nthreads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        st = C.verify_batch(pk[:per_step], msg[: 64 * per_step], off[: per_step + 1], sg[:per_step], nthreads=threads)
    dt = time.perf_counter() - t0
    if not (st == expect[:per_step]).all():
        raise SystemExit("bench (reference arm): the oracle's statuses differ from the ones expected by construction")
    value = per_step * args.steps / dt
    sample = f"the first {per_step} signatures of the GPU arm's rank-0 batch (same seeds, same 1/64 invalid mix) per step, oracle/ref10_port.c on {threads} host threads"
    print(json.dumps({
        "impl": "reference", "metric": "verified Ed25519 sigs/sec", "value": value, "unit": "sigs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": f"cfg2: batched EdDSA verify_with_checks of 2^{args.log2n} random keys / 64-byte messages / signatures per GPU incl. SHA-512 challenge, 1/64 invalid",
                   "sigs_per_step": per_step, "same_batch_as_gpu_arm": True,
                   "note": "CPU port of the reference's path (kyber-rs is Rust; no Rust toolchain in this image); it restates the reference's algorithm (4 inversions + constant-time variable-base mult per verify), "
                           "which is ~3.4x slower per core than libsodium"},
        "cpu_baseline": {"value": value, "unit": "sigs/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "sigs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=20)
    ap.add_argument("--no-extras", action="store_true", help="headline only (configs 1, 3, 4, 5 and the stage measurements are skipped)")
    ap.add_argument("--msm-max-log2", type=int, default=26)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the statuses of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    # Everything except the final JSON line goes to stderr: libraries (NCCL prints its version banner
    # on stdout when NCCL_DEBUG is set) must not pollute the one-line contract.
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")      # host-side waits that must not occupy the other ranks' GPUs
    kb = importlib.import_module("kyber-rs_b200")
    from helpers import load_c_oracle

    ctx = kb.Context(local_rank)
    dev = torch.device("cuda", local_rank)
    n = 1 << args.log2n
    C = load_c_oracle() if rank == 0 else None
    parity = []      # what this run compared, and against what

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def host_barrier():
        if world > 1:
            dist.barrier(group=cpu_group)

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ok(ok: bool, what: str):
        t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        if not int(t.item()):
            die(what)

    def timed(fn, reps=3):
        """seconds per call: CUDA events on the launch stream around EVERY repetition, barrier + synchronize on both sides,
        the MEDIAN over the repetitions (a single 20 ms hiccup of the box would otherwise triple a 6 ms round), MAX over ranks"""
        fn(); torch.cuda.synchronize()
        reps = max(reps, 5)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        barrier()
        for a, b in ev:
            a.record()
            fn()
            b.record()
        barrier()
        torch.cuda.synchronize()
        ms = sorted(a.elapsed_time(b) for a, b in ev)
        return max_over_ranks(ms[len(ms) // 2]) * 1e-3

    # ---- integer-multiply roofline denominator ---------------------------------------------------------------------
    # The path's multiplier is IMAD.WIDE.U32 (32x32+64 -> 64); it issues on the "fmaheavy" pipe at 4 cycles per warp
    # instruction, i.e. 32 lanes/clk/SM.  The denominator is that ARCHITECTURAL rate at the GPU's maximum SM clock; the
    # measured streams of kb_probe_imad are reported next to it.
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    sm_max_mhz = float(peaks.get("sm_max_mhz", 1965.0))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    imad_peak = 32.0 * ctx.sm_count * sm_max_mhz * 1e6
    probe_wide_plain, _ = ctx.probe_imad(0, 1 << 14)
    probe_wide_chain, _ = ctx.probe_imad(2, 1 << 13)
    imad_peak_lo, _ = ctx.probe_imad(1, 1 << 14)
    fe_mul_rate, _ = ctx.probe_imad(3, 1 << 10)

    # ---- cfg2 inputs ---------------------------------------------------------------------------------------------------
    pk, msg, off, sig, expect = make_batch(ctx, n, rank)
    if rank == 0 and C.point_decode_ok(OFF_CURVE):
        die("the off-curve constant decodes")
    d_pk = torch.from_numpy(pk).to(dev)
    d_msg = torch.from_numpy(msg).to(dev)
    d_off = torch.from_numpy(off.view(np.int64)).to(dev)
    d_sig = torch.from_numpy(sig).to(dev)
    d_st = torch.empty(n, dtype=torch.uint8, device=dev)

    def step_dev():
        ctx.dev_verify(n, d_pk, d_msg, d_off, d_sig, d_st)

    for _ in range(max(args.warmup, 3)):
        step_dev()
    torch.cuda.synchronize()
    got = d_st.cpu().numpy()
    bad = np.nonzero(got != expect)[0]
    all_ok(bad.size == 0, f"rank {rank}: {bad.size} verify statuses differ from the expected ones, first at {bad[:5]}: got {got[bad[:5]]} want {expect[bad[:5]]}")
    parity.append({"what": "cfg2 verify statuses vs the statuses expected by construction (valid + nine invalid classes incl. off-curve R = status 7 and the §A1 quirk range)",
                   "items": n * world, "ranks": world, "statuses_seen": sorted(set(int(x) for x in np.unique(got)))})

    # ---- timed region: device-resident value -----------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launches
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for k in range(args.steps):
        step_dev()
        ev[k + 1].record()
    barrier()
    launches = ctx.launches - l0
    clocks = sampler.stop()
    total_ms = ev[0].elapsed_time(ev[-1])
    kernel_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    dumped = {}
    if args.dump_outputs and rank == 0:
        dumped["verify_status"] = d_st.cpu().numpy()
    # the two launches of a step one by one: events recorded by the library around each launch, read back after
    # every step (a second pass, so that the read-back's synchronisation stays out of the timed region above)
    ctx.verify_kernel_timing(True)
    k_prep_ms, k_main_ms = [], []
    for _ in range(args.steps):
        step_dev()
        a_ms, b_ms = ctx.last_verify_kernel_ms()
        k_prep_ms.append(a_ms)
        k_main_ms.append(b_ms)
    ctx.verify_kernel_timing(False)
    total_ms_max = max_over_ranks(total_ms)
    value = world * n * args.steps / (total_ms_max * 1e-3)

    # ---- e2e: ONE host batch of world * n signatures through the multi-device context, on rank 0 -------------------
    # (the other ranks wait on the host; their GPUs are idle and are driven by rank 0's kb_mctx)
    e2e_value, h2d, e2e_launches = None, None, None
    mctx = None
    if rank == 0:
        mctx = kb.MultiContext(list(range(world)))
        batches = [(pk, msg, off, sig, expect)] + [make_batch(ctx, n, r) for r in range(1, world)]
        big_pk = np.concatenate([b[0] for b in batches])
        big_msg = np.concatenate([b[1] for b in batches])
        big_off = (np.arange(world * n + 1, dtype=np.uint64) * np.uint64(64))
        big_sig = np.concatenate([b[3] for b in batches])
        big_expect = np.concatenate([b[4] for b in batches])
        del batches
        hp = [torch.from_numpy(x).pin_memory() for x in (big_pk, big_msg, big_off.view(np.int64), big_sig)]
        h_pk, h_msg, h_off, h_sig = [x.numpy() for x in hp]
        h_off = h_off.view(np.uint64)
        h_out_t = torch.empty(world * n, dtype=torch.uint8).pin_memory()
        h_out = h_out_t.numpy()
    host_barrier()
    if rank == 0:
        for _ in range(2):
            mctx.verify_batch(h_pk, h_msg, h_off, h_sig, out=h_out)
        ml0 = mctx.launches
        t0 = time.perf_counter()
        for _ in range(args.steps):
            mctx.verify_batch(h_pk, h_msg, h_off, h_sig, out=h_out)
        e2e_s = time.perf_counter() - t0
        e2e_launches = mctx.launches - ml0
        if args.dump_outputs:
            dumped["e2e_verify_status"] = h_out.copy()
        if not (h_out == big_expect).all():
            die("e2e statuses (multi-device context) differ from the expected ones")
        e2e_value = world * n * args.steps / e2e_s
        h2d = int(big_pk.nbytes + big_msg.nbytes + big_off.nbytes + big_sig.nbytes)
        parity.append({"what": "e2e: kb_mctx_verify_batch statuses of ONE host batch sharded over all GPUs vs expected", "items": n * world, "devices": world})
        del hp, h_out_t, big_pk, big_msg, big_sig
    host_barrier()

    # ---- CPU baseline on rank 0 (N = 1 only): the oracle's C port on the host cores, bounded prefix; at N > 1 a short
    # prefix is still checked against the oracle on rank 0
    cpu = None
    if rank == 0:
        if world == 1:
            cpu = cpu_verify_baseline(C, pk, msg, off, sig, got, budget_s=12.0, threads=host_cores())
            parity.append({"what": "cfg2 verify statuses vs oracle/ref10_port.c", "items": cpu["checked_items"]})
        else:
            m = 16384
            st = C.verify_batch(pk[:m], msg[:64 * m], off[:m + 1], sig[:m], nthreads=host_cores())
            if not (st == got[:m]).all():
                die("GPU statuses differ from the oracle on rank 0's prefix")
            parity.append({"what": "cfg2 verify statuses vs oracle/ref10_port.c (rank 0 prefix)", "items": m})
    host_barrier()

    extras, configs, stages = {}, {}, {}
    if not args.no_extras:
        import bench_configs

        env = dict(kb=kb, ctx=ctx, mctx=mctx, C=C, dev=dev, rank=rank, world=world, dist=dist, torch=torch, timed=timed, barrier=barrier, host_barrier=host_barrier,
                   max_over_ranks=max_over_ranks, all_ok=all_ok, die=die, parity=parity, imad_peak=imad_peak, hbm_peak=hbm_peak, d_pk=d_pk, d_sig=d_sig, d_msg=d_msg, d_off=d_off,
                   n=n, args=args, host_cores=host_cores(), xof=xof)
        configs, stages = bench_configs.run_all(env)

    if mctx is not None:
        mctx.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumped)
    kernel_s = statistics.mean(kernel_ms) * 1e-3
    achieved = n * IMAD_EQ_PER_VERIFY / kernel_s
    prep_s, main_s = statistics.mean(k_prep_ms) * 1e-3, statistics.mean(k_main_ms) * 1e-3
    traffic, traffic_src = None, None
    try:   # dram__bytes of the two launches, measured by ncu on THIS build and stored by tools/ncu_traffic.py
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_verify_traffic.json")))
        if tr.get("log2n") == args.log2n:
            traffic, traffic_src = int(tr["dram_bytes_per_step"]), tr.get("source")
    except (OSError, ValueError, KeyError):
        pass
    out = {
        "metric": "verified Ed25519 sigs/sec", "value": value, "unit": "sigs/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": f"cfg2: batched EdDSA verify_with_checks of 2^{args.log2n} random keys / 64-byte messages / signatures per GPU incl. SHA-512 challenge, 1/64 invalid",
                   "sigs_per_gpu": n, "l2_policy": "inputs (168 MiB per step) exceed the 126 MB L2; no explicit flush", "parallelism": f"index-sharded x{world}, no data-path collective",
                   "same_batch_as_reference_arm": True},
        "e2e": {"value": e2e_value, "unit": "sigs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(n * world),
                "how": f"rank 0: kb_mctx_verify_batch on ONE pinned host batch of {world} x 2^{args.log2n} signatures, sharded by index over {world} GPU(s) inside the library (one host thread per device, "
                       "two-stream chunked copy/compute overlap per device); wall clock around the calls", "gpu_launches": e2e_launches},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "imad", "achieved": achieved / 1e12, "peak": imad_peak / 1e12, "unit": "T IMAD-eq/s", "frac": achieved / imad_peak, "traffic": traffic, "traffic_source": traffic_src,
                     "note": "integer-multiply roofline (north_star): 154k 32x32->64 MAC-equivalents CHARGED per signature (SURVEY 8d: decompress A + 253-doubling Straus + compress) / CUDA-event step time; "
                             f"peak = ARCHITECTURAL IMAD.WIDE.U32 rate, 32 lanes/clk/SM x {ctx.sm_count} SMs x {sm_max_mhz:.0f} MHz (the fmaheavy pipe issues one warp instruction per 4 cycles). "
                             "The kernels EXECUTE fewer multiplies than charged (half-size scalars: 128 doublings, csrc/half.cuh): see `executed`",
                     "kernel": "one step = k_verify_half_prep (checks, decompress A and R, SHA-512, lattice step) + k_half_sort_count/scan/scatter (records ordered by loop length; timed with the main kernel) + k_verify_half_main (joint radix-4 table of A and R, ~65 steps of two doublings and one addition, 15-position comb, verdict)",
                     "kernels_ms": {"k_verify_half_prep": prep_s * 1e3, "k_verify_half_main": main_s * 1e3, "timed_steps": len(k_main_ms),
                                    "how": "cudaEventRecord on the launch stream around each launch (kb_verify_kernel_times), averaged over a second pass of the same steps"},
                     "executed": {"imad_wide_per_sig": {"k_verify_half_prep": EXEC_PREP_PER_VERIFY, "k_verify_half_main": EXEC_MAIN_PER_VERIFY},
                                  "frac_step": n * (EXEC_PREP_PER_VERIFY + EXEC_MAIN_PER_VERIFY) / kernel_s / imad_peak,
                                  "frac_k_verify_half_main": n * EXEC_MAIN_PER_VERIFY / main_s / imad_peak,
                                  "frac_k_verify_half_prep": n * EXEC_PREP_PER_VERIFY / prep_s / imad_peak},
                     "probes_T_per_s": {"imad_lo32": imad_peak_lo / 1e12, "imad_wide_plain": probe_wide_plain / 1e12, "imad_wide_carry_chain": probe_wide_chain / 1e12, "fe_mul_as_imad_wide": fe_mul_rate * 73.0 / 72.0 / 1e12}},
        "roofline_hbm": {"bound": "hbm", "achieved": n * ALG_BYTES_PER_SIG / kernel_s / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": n * ALG_BYTES_PER_SIG / kernel_s / 1e9 / hbm_peak,
                         "note": "161 algorithmic bytes per signature; the path is integer-pipe bound, not HBM bound (peak: MEASURED_PEAKS.json)" if peaks else "peak: B200_PROFILING.md fallback"},
        "cpu_baseline": cpu,
        "parity_checked": parity,
        "configs": configs,
        "configs_timing": "every configs / stages entry: CUDA events on the launch stream around each repetition, median of >= 5 repetitions after one warm-up call, max over ranks",
        "stages": stages,
        "extras": extras,
    }
    os.write(real_stdout, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
