"""Timing of the batched aggregate verifier (ripp_tipp_verify_aggregate_batch, csrc/verify_batch.cuh) against a loop of
single ripp_tipp_verify_aggregate calls on the same aggregates.  One JSON line per measurement:

  batch_vs_loop  K = 1, 8, 32 aggregates of 2^12 proofs each (distinct permutations of one seeded instance, one vk, one
                 SRS): host clock around one batch call and around K sequential single calls (both end in a
                 synchronise), alternated in this call; medians of --reps runs after one warm-up of each; the ratio
                 loop / batch.  Every status is checked (all OK).
  split          one extra batch call at the largest K under torch.profiler: device time per step (subgroup checks,
                 G1 scalings and sums, GT folds, pairing equations) from the kernel records, and host_ms = the median
                 batch time minus the kernel time (host parsing, Fiat-Shamir chains, staging and copies).
device and power_limit_w are read in the same call.

Usage: python tools/time_verify_aggregate.py [--reps 5] [--ks 1,8,32] [--out verify_aggregate.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from ripp_b200 import _lib, synth  # noqa: E402

STEPS = {
    "subgroup": ("k_subgroup_check", "k_gt_check18"),
    "g1": ("k_input_column_ip_batch", "k_scale", "k_aff_seg_sum"),
    "gt_folds": ("k_gt_pow", "k_reduce6"),
    "equations": ("k_miller6", "k_groth16_check6"),
}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out)
    except Exception:
        power = None
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ks", default="1,8,32")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ks = [int(k) for k in args.ks.split(",")]
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this tool measures on the device only")
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
    n = 1 << 12
    t = synth.tipp_instance_dev(ctx, n)
    a, b, c = t["a"].download((n, 24)), t["b"].download((n, 48)), t["c"].download((n, 24))
    rng = np.random.default_rng(1)
    aggs = []
    for k in range(max(ks)):
        perm = np.arange(n) if k == 0 else rng.permutation(n)
        pa, pb, pc = ctx.to_device(a[perm]), ctx.to_device(b[perm]), ctx.to_device(c[perm])
        proof = ctx.tipp_aggregate_dev(t["srs_g1"], t["srs_g2"], pa, pb, pc, n)
        aggs.append((np.ascontiguousarray(t["inputs"][perm]), proof))
    vsrs, vk = t["vsrs"], t["vk"]

    def batch(members):
        st = ctx.tipp_verify_aggregate_batch(vsrs, vk, [r for r, _ in members], [p for _, p in members])
        assert list(st) == [0] * len(members), list(st)

    def loop(members):
        for r, p in members:
            assert ctx.tipp_verify_aggregate(vsrs, vk, r, p)

    med = {}
    for K in ks:
        members = aggs[:K]
        batch(members)
        loop(members)
        tb, tl = [], []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            batch(members)
            tb.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            loop(members)
            tl.append(time.perf_counter() - t0)
        med[K] = statistics.median(tb)
        emit({"what": "batch_vs_loop", "k": K, "n": n, "batch_ms": 1e3 * med[K], "loop_ms": 1e3 * statistics.median(tl),
              "loop_over_batch": statistics.median(tl) / med[K], "reps": args.reps})

    K = max(ks)
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        batch(aggs[:K])
        torch.cuda.synchronize()
    split = {s: 0.0 for s in STEPS}
    total = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        for s, keys in STEPS.items():
            if any(ev.name.startswith(k) or k in ev.name for k in keys):
                split[s] += us / 1e3
                total += us / 1e3
                break
    emit({"what": "split", "k": K, "n": n, **{s + "_ms": v for s, v in split.items()}, "kernels_ms": total,
          "host_ms": 1e3 * med[K] - total})
    ctx.close()


if __name__ == "__main__":
    main()
