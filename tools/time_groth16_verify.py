"""Timing of Groth16 verification with one verdict per proof (csrc/groth16.cu).  One JSON line per measurement:

  prepare_vk        m = 5: device-event time of ripp_groth16_prepare_vk_dev (e(alpha, beta), -gamma, -delta, IC_0, the
                    m fixed-base tables)
  verify_batch_dev  n = 2^4, 2^8, 2^12, 2^16 proofs with m = 5, and 2^12 with m = 1: device-event time of
                    ripp_groth16_verify_batch_dev (proofs and inputs resident), proofs/s, and the per-class split of
                    ripp_ctx_timing from one extra run (scale = prepare_inputs, miller, final_exp = final
                    exponentiation + compare)
  serialized        2^12 and 2^16 compressed records in host memory: host clock around
                    ripp_groth16_verify_serialized (H2D, decode, verify, D2H of the statuses), proofs/s
  rlc_vs_batch      m = 5 at 2^12 and 2^16, all valid and with 41 false proofs (C + G): ripp_groth16_verify_rlc_dev and
                    ripp_groth16_verify_batch_dev on the same proofs, alternated in this call (device events), the
                    ratio, n_rechecked, and the class split of one extra run of each (scale = the r_i A_i, r_i C_i
                    scalings + C_s + P_s / prepare_inputs, miller, final_exp, other = scalars, gather, scatter; the
                    fallback's kernels count in their own classes, fallback_ms = the 41-false time minus the
                    all-valid time)
  rlc_serialized    2^12 and 2^16 compressed records: host clock around ripp_groth16_verify_rlc_serialized and
                    ripp_groth16_verify_serialized, alternated
Every shape is warmed up once; times are medians of --reps runs.  Every verdict is checked.
device and power_limit_w are read in the same call.

  --rlc-only        only the rlc_vs_batch lines (with --sweep)
  --sweep S[:KP],.. the rlc_vs_batch lines once per segment size S (RIPP_B200_G16_RLC_SEG), optionally with the
                    pairs per six-lane group pinned to KP (RIPP_B200_M6_KP), each in a subprocess (both switches are
                    read once per process)

Usage: python tools/time_groth16_verify.py [--reps 5] [--rlc-only] [--sweep 58,118,18:1]
"""
import argparse
import json
import os
import random
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from oracle import serde_cases as SC  # noqa: E402
from ripp_b200 import _lib, codec, synth  # noqa: E402
from tools.time_deserialize import card  # noqa: E402


def instance(ctx, n, m, seed=0, nfalse=0):
    vk, ic, proofs, inputs = synth.groth16_scalars(n, m, seed)
    proofs = list(proofs)
    for i in random.Random(seed).sample(range(n), nfalse):  # C + G: false
        a_, b_, c_ = proofs[i]
        proofs[i] = (a_, b_, (c_ + 1) % codec.R)
    g1 = synth._gen_dev(ctx, 1, [vk["alpha"]] + ic).download((m + 2, 24))
    g2 = synth._gen_dev(ctx, 2, [vk["beta"], vk["gamma"], vk["delta"]]).download((3, 48))
    vk_words = np.concatenate([g1[0], g2[0], g2[1], g2[2]] + [g1[1 + j] for j in range(m + 1)])
    a = synth._gen_dev(ctx, 1, [p[0] for p in proofs])
    b = synth._gen_dev(ctx, 2, [p[1] for p in proofs])
    c = synth._gen_dev(ctx, 1, [p[2] for p in proofs])
    x = ctx.to_device(codec.fr_vec_enc([v for row in inputs for v in row]))
    xb = b"".join(v.to_bytes(32, "little") for row in inputs for v in row)
    return vk_words, a, b, c, x, xb


def events(ctx, fn, reps):
    stream = torch.cuda.ExternalStream(ctx.stream)
    ms = []
    for r in range(reps + 1):  # the first pass loads the modules and grows the scratch buffers
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        if r:
            ms.append(e0.elapsed_time(e1))
    return float(np.median(ms))


def alternate(ctx, fns, reps):
    """Median device-event time of each fn, the fns run in turn, reps rounds after one warm-up round."""
    stream = torch.cuda.ExternalStream(ctx.stream)
    ms = [[] for _ in fns]
    for r in range(reps + 1):
        for k, fn in enumerate(fns):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            if r:
                ms[k].append(e0.elapsed_time(e1))
    return [float(np.median(v)) for v in ms]


def split(ctx, fn):
    ctx.set_timing(True)
    ctx.timing()
    fn()
    out = {k: round(v[0], 3) for k, v in ctx.timing().items() if v[1]}
    ctx.set_timing(False)
    return out


SEED = bytes(range(32))


def rlc_lines(ctx, emit, reps, serialized):
    m = 5
    for lg in (12, 16):
        n = 1 << lg
        base_ms = None
        for nfalse in (0, 41):
            vk_words, a, b, c, x, xb = instance(ctx, n, m, nfalse=nfalse)
            pvk = ctx.alloc(ctx.groth16_pvk_bytes(m))
            ctx.groth16_prepare_vk_dev(vk_words, m, pvk)
            out_b, out_r = ctx.alloc(n), ctx.alloc(n)
            nre = [0]

            def rlc():
                nre[0] = ctx.groth16_verify_rlc_dev(pvk, m, x, a, b, c, n, SEED, out_r)

            t_batch, t_rlc = alternate(ctx, [lambda: ctx.groth16_verify_batch_dev(pvk, m, x, a, b, c, n, out_b), rlc], reps)
            vb, vr = out_b.download(n, dtype=np.uint8), out_r.download(n, dtype=np.uint8)
            assert (vb == vr).all() and int(vb.sum()) == n - nfalse, "verdicts differ"
            line = {"what": "rlc_vs_batch", "n": n, "m": m, "false": nfalse, "batch_ms": round(t_batch, 3), "rlc_ms": round(t_rlc, 3),
                    "rlc_over_batch": round(t_rlc / t_batch, 3), "n_rechecked": nre[0],
                    "seg": os.environ.get("RIPP_B200_G16_RLC_SEG", "default"), "kp": os.environ.get("RIPP_B200_M6_KP", "auto"),
                    "rlc_class_ms": split(ctx, rlc),
                    "batch_class_ms": split(ctx, lambda: ctx.groth16_verify_batch_dev(pvk, m, x, a, b, c, n, out_b))}
            if nfalse == 0:
                base_ms = t_rlc
            else:
                line["fallback_ms"] = round(t_rlc - base_ms, 3)
            emit(line)
            if serialized and nfalse == 0:
                data = SC.proof_records(a.download((n, 24)), b.download((n, 48)), c.download((n, 24)), True)
                t = [[], []]
                for r in range(reps + 1):
                    for k in range(2):
                        t0 = time.perf_counter()
                        if k:
                            st, nv, nr = ctx.groth16_verify_rlc_serialized(pvk, m, xb, data, n, True, SEED)
                        else:
                            st, nv = ctx.groth16_verify_serialized(pvk, m, xb, data, n, True)
                        t1 = time.perf_counter()
                        assert nv == n
                        if r:
                            t[k].append(1e3 * (t1 - t0))
                emit({"what": "rlc_serialized", "n": n, "m": m, "serialized_ms": round(float(np.median(t[0])), 3),
                      "rlc_serialized_ms": round(float(np.median(t[1])), 3)})
            for buf in (a, b, c, x, pvk, out_b, out_r):
                buf.free()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rlc-only", action="store_true")
    ap.add_argument("--sweep", default="")
    args = ap.parse_args()
    if args.sweep:
        for item in args.sweep.split(","):
            seg, _, kp = item.partition(":")
            env = dict(os.environ, RIPP_B200_G16_RLC_SEG=seg)
            if kp:
                env["RIPP_B200_M6_KP"] = kp
            subprocess.run([sys.executable, os.path.abspath(__file__), "--reps", str(args.reps), "--rlc-only"], env=env, check=True)
        return
    ctx = _lib.Context(0)
    name, power = card()
    base = {"device": name, "power_limit_w": power}

    def emit(d):
        print(json.dumps(dict(base, **d)), flush=True)

    if args.rlc_only:
        rlc_lines(ctx, emit, args.reps, False)
        ctx.close()
        return

    insts = {}
    for lg, m in ((4, 5), (8, 5), (12, 5), (16, 5), (12, 1)):
        n = 1 << lg
        vk_words, a, b, c, x, xb = insts[(lg, m)] = instance(ctx, n, m)
        pvk = ctx.alloc(ctx.groth16_pvk_bytes(m))
        if (lg, m) == (4, 5):
            emit({"what": "prepare_vk", "m": m, "ms": round(events(ctx, lambda: ctx.groth16_prepare_vk_dev(vk_words, m, pvk), args.reps), 3),
                  "pvk_bytes": ctx.groth16_pvk_bytes(m)})
        ctx.groth16_prepare_vk_dev(vk_words, m, pvk)
        out = ctx.alloc(n)
        ms = events(ctx, lambda: ctx.groth16_verify_batch_dev(pvk, m, x, a, b, c, n, out), args.reps)
        assert out.download(n, dtype=np.uint8).all(), "a valid proof was rejected"
        ctx.set_timing(True)
        ctx.timing()
        ctx.groth16_verify_batch_dev(pvk, m, x, a, b, c, n, out)
        split = {k: round(v[0], 3) for k, v in ctx.timing().items() if v[1]}
        ctx.set_timing(False)
        emit({"what": "verify_batch_dev", "n": n, "m": m, "ms": round(ms, 3), "proofs_per_s": round(n / ms * 1e3),
              "class_ms": split})
        if m == 5 and lg in (12, 16):
            data = SC.proof_records(a.download((n, 24)), b.download((n, 48)), c.download((n, 24)), True)
            t = []
            for r in range(args.reps + 1):
                t0 = time.perf_counter()
                st, nv = ctx.groth16_verify_serialized(pvk, m, xb, data, n, True)
                t1 = time.perf_counter()
                assert nv == n
                if r:
                    t.append(1e3 * (t1 - t0))
            ms = float(np.median(t))
            emit({"what": "serialized_compressed", "n": n, "m": m, "ms": round(ms, 3), "proofs_per_s": round(n / ms * 1e3)})
        for buf in (a, b, c, x, pvk, out):
            buf.free()
        del insts[(lg, m)]
    rlc_lines(ctx, emit, args.reps, True)
    ctx.close()


if __name__ == "__main__":
    main()
