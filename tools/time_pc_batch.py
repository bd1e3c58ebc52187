"""Timing of the batched polynomial commitments (ripp_pc_commit_batch_dev, ripp_pc_open_batch_dev; csrc/pc_batch.cuh)
and of the batched verifier (ripp_pc_verify_batch; csrc/pc_verify_batch.cuh) against K sequential ripp_pc_commit_dev /
ripp_pc_open_dev / ripp_pc_verify calls on the same inputs.  One JSON line per measurement:

  batch_vs_loop  both kinds, univariate polynomials of 2^10, 2^12 and 2^16 coefficients (the univariate wrappers'
                 bivariate shapes), K = 1, 8, 32 polynomials (seeded, full length, random points): host clock around one
                 batch call and around K sequential single calls (all synchronous), commit, open and verify separately,
                 alternated, medians of --reps runs after one warm-up of each; the ratio batch / loop.  The bytes of every
                 batch run are compared with the loop's; verify checks the K openings just made (every status accepted,
                 equal to the loop's verdicts).
  split          one open and one verify at K = 32 and --split-coeffs coefficients per kind under torch.profiler: device
                 time by kernel kind.
device and power_limit_w are read in the same call.

Usage: python tools/time_pc_batch.py [--reps 5] [--coeffs 10,12,16] [--ks 1,8,32] [--split-coeffs 12] [--out pc_batch.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from ripp_b200 import _lib, codec, synth  # noqa: E402
from ripp_b200 import poly_commit as PC  # noqa: E402
from ripp_b200.ip_proofs import AGG_OK, AGG_REJECTED, vsrs_enc  # noqa: E402

KINDS = {
    "pairing": ("k_miller6", "k_reduce6", "k_final_exp", "k_miller18", "k_reduce18", "k_groth16_check"),
    "msm": ("k_msm_",),
    "fold": ("k_fold",),
    "pc_scalar": ("k_pc_",),
    "gather": ("k_gather",),
    "gt": ("k_gt_",),
    "subgroup": ("k_subgroup",),
    "g1_scale_sum": ("k_scale", "k_aff_seg_sum", "k_normalize"),
}
R = codec.R


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out)
    except Exception:
        power = None
    return name, power


def keys(ctx, kind, lg):
    """The univariate wrappers' keys for polynomials of 2^lg coefficients: (first, m, second, n, h_beta_powers, vsrs)."""
    if kind == _lib.PC_TRUSTED:
        xd, yd = PC.UnivariatePolynomialCommitment.bivariate_degrees((1 << lg) - 1)
        srs = PC.BivariatePolynomialCommitment.setup(xd, yd, 12345, 67890, ctx)
        return srs["kzg"][0], yd + 1, srs["ck"][0], xd + 1, srs["h_beta_powers"][0], vsrs_enc(srs["v_srs"])
    xd, yd = PC.TransparentUnivariatePolynomialCommitment.bivariate_degrees((1 << lg) - 1)
    return synth.g1_points_dev(ctx, "tpcb-1", yd + 1), yd + 1, synth.g2_points_dev(ctx, "tpcb-2", xd + 1), xd + 1, None, None


def words(seed, count):
    w = np.random.default_rng(seed).integers(0, 1 << 32, size=(count, 8), dtype=np.uint32)
    w[:, 7] %= np.uint32(R >> 224)
    return w


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--coeffs", default="10,12,16")
    ap.add_argument("--ks", default="1,8,32")
    ap.add_argument("--split-coeffs", type=int, default=12)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
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
    kmax = max(int(x) for x in args.ks.split(","))
    for kind in (_lib.PC_TRUSTED, _lib.PC_TRANSPARENT):
        kname = "trusted" if kind == _lib.PC_TRUSTED else "transparent"
        for lg in (int(x) for x in args.coeffs.split(",")):
            first, m, second, n, g2, vsrs = keys(ctx, kind, lg)
            N = n * m
            pool = [ctx.to_device(words(1000 * lg + i, N)) for i in range(kmax)]
            rng = np.random.default_rng(lg)
            zs = [codec.fr_enc(int(rng.integers(1, 1 << 62)) % R) for _ in range(kmax)]
            ws = [codec.fr_enc(int(rng.integers(1, 1 << 62)) % R) for _ in range(kmax)]
            for K in (int(x) for x in args.ks.split(",")):
                bufs, lens, xs, ys = pool[:K], [N] * K, np.stack(zs[:K]), np.stack(ws[:K])
                yb = ctx.alloc(K * n * 96)
                ysingle = [ctx.alloc(n * 96) for _ in range(K)]

                def commit_batch():
                    return ctx.pc_commit_batch_dev(first, m, second, n, bufs, lens, yb).tolist()

                def commit_loop():
                    return [ctx.pc_commit_dev(first, m, second, n, bufs[i], N, ysingle[i]).tolist() for i in range(K)]

                def open_batch():
                    p, e = ctx.pc_open_batch_dev(kind, first, m, second, n, g2, bufs, lens, yb, xs, ys)
                    return p, e.tolist()

                def open_loop():
                    r = [ctx.pc_open_dev(kind, first, m, second, n, g2, bufs[i], N, ysingle[i], xs[i], ys[i]) for i in range(K)]
                    return [p for p, _ in r], [e.tolist() for _, e in r]

                opened = {}

                def verify_batch():
                    coms, (proofs, evs) = opened["v"]
                    return ctx.pc_verify_batch(kind, vsrs, first, m, second, n, coms, xs, ys, evs, proofs).tolist()

                def verify_loop():
                    coms, (proofs, evs) = opened["v"]
                    return [AGG_OK if ctx.pc_verify(kind, vsrs, first, m, second, n, coms[i], xs[i], ys[i], evs[i], proofs[i])
                            else AGG_REJECTED for i in range(K)]

                for what, batch, loop in (("commit", commit_batch, commit_loop), ("open", open_batch, open_loop),
                                          ("verify", verify_batch, verify_loop)):
                    if what == "verify":
                        proofs, evs = open_batch()
                        opened["v"] = (np.array(commit_batch(), dtype=np.uint32), (proofs, np.array(evs, dtype=np.uint32)))
                    want = loop()
                    if what == "verify":
                        assert want == [AGG_OK] * K, "an honest opening was rejected"
                    assert batch() == want, "batch bytes differ from the single calls (%s %s 2^%d, K = %d)" % (kname, what, lg, K)
                    tb, tl = [], []
                    for _ in range(args.reps):
                        t0 = time.perf_counter()
                        got = batch()
                        tb.append(time.perf_counter() - t0)
                        assert got == want, "batch bytes differ from the single calls"
                        t0 = time.perf_counter()
                        assert loop() == want
                        tl.append(time.perf_counter() - t0)
                    mb, ml = statistics.median(tb), statistics.median(tl)
                    emit({"what": "batch_vs_loop", "kind": kname, "op": what, "coeffs": N, "n": n, "m": m, "k": K,
                          "batch_ms": 1e3 * mb, "loop_ms": 1e3 * ml, "batch_over_loop": mb / ml, "bytes_equal": True,
                          "reps": args.reps})
            for b in pool:
                b.free()

    from torch.profiler import ProfilerActivity, profile

    for kind in (_lib.PC_TRUSTED, _lib.PC_TRANSPARENT):
        K, lg = 32, args.split_coeffs
        first, m, second, n, g2, vsrs = keys(ctx, kind, lg)
        bufs = [ctx.to_device(words(77 + i, n * m)) for i in range(K)]
        yb = ctx.alloc(K * n * 96)
        xs = np.stack([codec.fr_enc(3 + i) for i in range(K)])
        ys = np.stack([codec.fr_enc(5 + i) for i in range(K)])
        coms = np.array(ctx.pc_commit_batch_dev(first, m, second, n, bufs, [n * m] * K, yb), dtype=np.uint32)
        proofs, evs = ctx.pc_open_batch_dev(kind, first, m, second, n, g2, bufs, [n * m] * K, yb, xs, ys)
        ctx.pc_verify_batch(kind, vsrs, first, m, second, n, coms, xs, ys, evs, proofs)
        ops = {"open": lambda: ctx.pc_open_batch_dev(kind, first, m, second, n, g2, bufs, [n * m] * K, yb, xs, ys),
               "verify": lambda: ctx.pc_verify_batch(kind, vsrs, first, m, second, n, coms, xs, ys, evs, proofs)}
        for op, run in ops.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run()
                torch.cuda.synchronize()
            split = {s: 0.0 for s in KINDS}
            split["other"] = 0.0
            for ev in prof.events():
                if ev.device_type != torch.autograd.DeviceType.CUDA:
                    continue
                ms = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
                kk = next((s for s, names in KINDS.items() if any(x in ev.name for x in names)), "other")
                split[kk] += ms
            emit({"what": "split", "kind": "trusted" if kind == _lib.PC_TRUSTED else "transparent", "op": op, "coeffs": n * m,
                  "k": K, **{s + "_ms": v for s, v in split.items()}, "kernels_ms": sum(split.values())})
    ctx.close()


if __name__ == "__main__":
    main()
