"""Timing of Groth16 verification with one verdict per proof (csrc/groth16.cu).  One JSON line per measurement:

  prepare_vk        m = 5: device-event time of ripp_groth16_prepare_vk_dev (e(alpha, beta), -gamma, -delta, IC_0, the
                    m fixed-base tables)
  verify_batch_dev  n = 2^4, 2^8, 2^12, 2^16 proofs with m = 5, and 2^12 with m = 1: device-event time of
                    ripp_groth16_verify_batch_dev (proofs and inputs resident), proofs/s, and the per-class split of
                    ripp_ctx_timing from one extra run (scale = prepare_inputs, miller, final_exp = final
                    exponentiation + compare)
  serialized        2^12 and 2^16 compressed records in host memory: host clock around
                    ripp_groth16_verify_serialized (H2D, decode, verify, D2H of the statuses), proofs/s
Every shape is warmed up once; times are medians of --reps runs.  All proofs are valid and every verdict is checked.
device and power_limit_w are read in the same call.

Usage: python tools/time_groth16_verify.py [--reps 5]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from oracle import serde_cases as SC  # noqa: E402
from ripp_b200 import _lib, codec, synth  # noqa: E402
from tools.time_deserialize import card  # noqa: E402


def instance(ctx, n, m, seed=0):
    vk, ic, proofs, inputs = synth.groth16_scalars(n, m, seed)
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    ctx = _lib.Context(0)
    name, power = card()
    base = {"device": name, "power_limit_w": power}

    def emit(d):
        print(json.dumps(dict(base, **d)), flush=True)

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
    ctx.close()


if __name__ == "__main__":
    main()
