"""Timing of the lock-step batch prover (ripp_tipp_aggregate_batch_dev, csrc/aggregate_batch.cuh) against K sequential
ripp_tipp_aggregate_dev calls on the same batches.  One JSON line per measurement:

  batch_vs_loop  n = 2^6, 2^8, 2^10, 2^12 proofs per batch, K = 1, 8, 32 batches (distinct permutations of one seeded
                 instance of 2^12 proofs, one SRS): host clock around one batch call and around K sequential single calls
                 (both end in a synchronise), alternated, medians of --reps runs after one warm-up of each; the ratio
                 loop / batch.  The bytes of every batch run are compared with the loop's.
  phases         one batch call at K = 32 and --phase-n, in a child process with RIPP_B200_TRACE=1: host wall clock of
                 the prologue (queued), the rounds (products, challenges, folds) and the openings (quotients, MSMs).
  split          the same call under torch.profiler: device time by kernel kind.
device and power_limit_w are read in the same call.

Usage: python tools/time_aggregate_batch.py [--reps 5] [--ns 6,8,10,12] [--ks 1,8,32] [--phase-n 10] [--out agg_batch.jsonl]
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from ripp_b200 import _lib, synth  # noqa: E402

KINDS = {
    "pairing": ("k_miller6", "k_reduce6", "k_final_exp", "k_miller18", "k_reduce18"),
    "msm": ("k_msm_",),
    "fold": ("k_fold",),
    "scale": ("k_scale", "k_fr_powers", "k_gather"),
}
NPOOL = 1 << 12


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out)
    except Exception:
        power = None
    return name, power


class Pool:
    def __init__(self, ctx):
        self.ctx = ctx
        t = synth.tipp_instance_dev(ctx, NPOOL)
        self.t = t
        self.h = t["a"].download((NPOOL, 24)), t["b"].download((NPOOL, 48)), t["c"].download((NPOOL, 24))
        self.rng = np.random.default_rng(1)

    def batches(self, K, n):
        """K distinct batches of n proofs: device buffers of all K n proofs and of each batch alone."""
        idx = [self.rng.permutation(NPOOL)[:n] for _ in range(K)]
        flat = np.concatenate(idx)
        allb = [self.ctx.to_device(x[flat]) for x in self.h]
        each = [[self.ctx.to_device(x[i]) for x in self.h] for i in idx]
        return allb, each


def child_phases(K, n):
    """One warm-up and one traced batch call (RIPP_B200_TRACE is read once per process)."""
    ctx = _lib.Context(0)
    pool = Pool(ctx)
    (a, b, c), _ = pool.batches(K, n)
    t = pool.t
    ctx.tipp_aggregate_batch_dev(t["srs_g1"], t["srs_g2"], a, b, c, K, n)
    print("=== traced call", file=sys.stderr, flush=True)
    t0 = time.perf_counter()
    ctx.tipp_aggregate_batch_dev(t["srs_g1"], t["srs_g2"], a, b, c, K, n)
    print("[total] %.3f ms" % (1e3 * (time.perf_counter() - t0)), file=sys.stderr, flush=True)
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ns", default="6,8,10,12")
    ap.add_argument("--ks", default="1,8,32")
    ap.add_argument("--phase-n", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures on the device only")
    if args.child:
        K, lg = (int(x) for x in args.child.split(","))
        return child_phases(K, 1 << lg)
    name, power = card()
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        rec.update(device=name, power_limit_w=power)
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    ctx = _lib.Context(0)
    pool = Pool(ctx)
    s1, s2 = pool.t["srs_g1"], pool.t["srs_g2"]
    for lg in (int(x) for x in args.ns.split(",")):
        n = 1 << lg
        for K in (int(x) for x in args.ks.split(",")):
            if K * n > (1 << 20):
                continue
            (a, b, c), each = pool.batches(K, n)

            def batch():
                r = ctx.tipp_aggregate_batch_dev(s1, s2, a, b, c, K, n)
                ctx.sync()
                return r

            def loop():
                r = [ctx.tipp_aggregate_dev(s1, s2, x, y, z, n) for x, y, z in each]
                ctx.sync()
                return r

            want = loop()
            assert batch() == want
            tb, tl = [], []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                got = batch()
                tb.append(time.perf_counter() - t0)
                assert got == want, "batch bytes differ from the single calls (n = %d, K = %d)" % (n, K)
                t0 = time.perf_counter()
                assert loop() == want
                tl.append(time.perf_counter() - t0)
            mb, ml = statistics.median(tb), statistics.median(tl)
            emit({"what": "batch_vs_loop", "n": n, "k": K, "batch_ms": 1e3 * mb, "loop_ms": 1e3 * ml, "loop_over_batch": ml / mb,
                  "batch_over_loop": mb / ml, "bytes_equal": True, "reps": args.reps})

    # phases (host trace in a child process) and the device split of one K = 32 call
    K, lg = 32, args.phase_n
    env = dict(os.environ, RIPP_B200_TRACE="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "%d,%d" % (K, lg)], env=env, capture_output=True,
                       text=True, timeout=1800)
    err = r.stderr.split("=== traced call", 1)[-1]
    pro = sum(float(x) for x in re.findall(r"aggregate batch prologue .*? ([\d.]+) ms", err))
    rounds = [float(x) for x in re.findall(r"aggregate batch round n' = \d+ ([\d.]+) ms", err)]
    openings = re.findall(r"aggregate batch openings ([\d.]+) ms", err)
    quot = re.findall(r"aggregate batch quotients \(host\) ([\d.]+) ms", err)
    total = re.findall(r"\[total\] ([\d.]+) ms", err)
    emit({"what": "phases", "n": 1 << lg, "k": K, "prologue_queued_ms": pro, "rounds_ms": sum(rounds), "round_ms": rounds,
          "openings_ms": float(openings[0]) if openings else None, "quotients_host_ms": float(quot[0]) if quot else None,
          "total_ms": float(total[0]) if total else None, "child_exit": r.returncode})

    from torch.profiler import ProfilerActivity, profile

    n = 1 << lg
    (a, b, c), _ = pool.batches(K, n)
    ctx.tipp_aggregate_batch_dev(s1, s2, a, b, c, K, n)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.tipp_aggregate_batch_dev(s1, s2, a, b, c, K, n)
        torch.cuda.synchronize()
    split = {s: 0.0 for s in KINDS}
    split["other"] = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        ms = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
        kind = next((s for s, keys in KINDS.items() if any(k in ev.name for k in keys)), "other")
        split[kind] += ms
    emit({"what": "split", "n": n, "k": K, **{s + "_ms": v for s, v in split.items()}, "kernels_ms": sum(split.values())})
    ctx.close()


if __name__ == "__main__":
    main()
