"""Timing of the polynomial-commitment entry points (ripp_pc_commit_dev, ripp_pc_open_dev, ripp_pc_verify;
csrc/poly_commit.cuh) at univariate degrees 2^16, 2^20 and 2^22 - 1 (n x m = 2^16, 2^20, 2^22 coefficients), trusted and
transparent.  One JSON line per measurement:

  new      host clock around commit, open and verify with the coefficients already on the device (each call ends in a
           synchronise); medians of --reps runs after one warm-up.
  old      the composition the Python layer ran before on the same device buffers: one ripp_msm_g1_dev per Y polynomial
           (each with its synchronise and download) plus the pairing product; the open's y_eval combination and KZG
           quotient in Python big-int arithmetic from the coefficients as ints (their decoding is not timed: the old
           API took ints), then the same MSMs and resident provers.  Medians of --old-reps runs.  The old and new
           commitments and proofs are compared byte for byte on every size.
  split    one commit and one open under torch.profiler: device time by kernel kind (msm, pairing, fold / scale of the
           GIPA / TIPA rounds, the new Fr kernels k_pc_* and k_fr_power_seq, other).
device and power_limit_w are read in the same call.

Usage: python tools/time_poly_commit.py [--reps 3] [--old-reps 1] [--logs 16,20,22] [--out pc.jsonl]
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

R = codec.R
RINV = pow(1 << 256, -1, R)
KINDS = {
    "pc_fr": ("k_pc_", "k_fr_power_seq"),
    "msm": ("k_msm_",),
    "pairing": ("k_miller6", "k_reduce6", "k_final_exp", "k_miller18", "k_reduce18"),
    "gipa_fold_scale": ("k_fold", "k_scale", "k_fr_powers", "k_gather", "k_fr_dot"),
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


def rand_fr_words(rng, n):
    """n canonical Fr (< r: the top word stays below r's), used directly as Montgomery words."""
    w = rng.integers(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    w[:, 7] %= 0x73EDA753
    return w


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def powers(s, n):
    out, cur = [], 1
    for _ in range(n):
        out.append(cur)
        cur = cur * s % R
    return out


def old_commit(ctx, first, m, second, n, c):
    coms = np.zeros((n, 24), dtype=np.uint32)
    out = ctx.alloc(96)
    for i in range(n):
        ctx.msm_g1_dev(first, c.ptr + i * m * 32, m, out)
        ctx.sync()
        coms[i] = out.download(24)
    d = ctx.to_device(coms)
    gt = ctx.alloc(576)
    ctx.pairing_ip_dev(d, second, n, gt)
    ctx.sync()
    return gt.download(144), d


def old_msm(ctx, bases, vals):
    sc = ctx.to_device(codec.fr_vec_enc(vals))
    out = ctx.alloc(96)
    ctx.msm_g1_dev(bases, sc, len(vals), out)
    ctx.sync()
    return codec.ser_g1(codec.g1_dec(out.download(24)))


def old_open(ctx, kind, first, m, second, n, srs_g2, ints, y_coms, x, y):
    px = powers(x, n)
    y_eval = [0] * m
    for i in range(n):  # mod.rs:221-241 as the Python layer did it
        p, row = px[i], ints[i * m:(i + 1) * m]
        for j, cj in enumerate(row):
            y_eval[j] = (y_eval[j] + p * cj) % R
    ye = old_msm(ctx, first, y_eval)
    b = ctx.to_device(codec.fr_vec_enc(px))
    if kind == _lib.PC_TRUSTED:
        ip = ctx.tipa_prove_dev(_lib.GIPA_MULTIEXP_SSM, None, srs_g2, y_coms, b, second, None, n)
        q = PC.quotient_by_linear(y_eval, y)
        return ip + ye + old_msm(ctx, first, q + [0] * (m - len(q)))
    ip2 = ctx.gipa_prove_dev(_lib.GIPA_MULTIEXP_SSM, y_coms, b, second, None, n)[0]
    a1, b1 = ctx.to_device(codec.fr_vec_enc(y_eval)), ctx.to_device(codec.fr_vec_enc(powers(y, m)))
    return ip2 + ye + ctx.gipa_prove_dev(_lib.GIPA_SCALAR_SSM_G1, a1, b1, first, None, m)[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--old-reps", type=int, default=1)
    ap.add_argument("--logs", default="16,20,22")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_poly_commit.py measures the GPU: no CUDA device")
    name, power = card()
    out = open(a.out, "a") if a.out else None

    def emit(rec):
        rec.update(device=name, power_limit_w=power)
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    ctx = _lib.Context(0)
    rng = np.random.default_rng(7)
    alpha, beta = 0x1234567 ** 5 % R, 0x7654321 ** 5 % R
    for lg in [int(v) for v in a.logs.split(",")]:
        degree = (1 << lg) - 1
        for kind in (_lib.PC_TRUSTED, _lib.PC_TRANSPARENT):
            if kind == _lib.PC_TRUSTED:
                U = PC.UnivariatePolynomialCommitment
                key = U.setup(degree, alpha, beta, ctx)
                xd, yd = U.degrees_from_srs(key)
                first, second, srs_g2 = key["kzg"][0], key["ck"][0], key["h_beta_powers"][0]
                verify = lambda cm, z, e, pf: U.verify(key["v_srs"], degree, cm, z, e, pf, ctx)  # noqa: E731
            else:
                U = PC.TransparentUnivariatePolynomialCommitment
                xd, yd = U.bivariate_degrees(degree)
                key = {"first": (synth.g1_points_dev(ctx, "tpc-ck1", yd + 1), yd + 1),
                       "second": (synth.g2_points_dev(ctx, "tpc-ck2", xd + 1), xd + 1)}
                first, second, srs_g2 = key["first"][0], key["second"][0], None
                verify = lambda cm, z, e, pf: U.verify(key, cm, z, e, pf, ctx)  # noqa: E731
            n, m = xd + 1, yd + 1
            words = rand_fr_words(rng, n * m)
            c = ctx.to_device(words)
            z = int(rng.integers(1, 1 << 62))
            kname = "trusted" if kind == _lib.PC_TRUSTED else "transparent"
            res = {}
            t_commit = timed(lambda: res.__setitem__("c", U.commit_dev(key, c, n * m, ctx)), a.reps)
            com, y_dev = res["c"]
            t_open = timed(lambda: res.__setitem__("o", U.open_dev(key, c, n * m, y_dev, z, ctx)), a.reps)
            proof, ev = res["o"]
            t_verify = timed(lambda: res.__setitem__("v", verify(com, z, ev, proof)), a.reps)
            assert res["v"], "the opening did not verify"
            emit({"what": "new", "kind": kname, "log_coeffs": lg, "x_degree": xd, "y_degree": yd, "commit_ms": t_commit,
                  "open_ms": t_open, "verify_ms": t_verify, "proof_bytes": len(proof)})

            t_oc = timed(lambda: res.__setitem__("oc", old_commit(ctx, first, m, second, n, c)), a.old_reps)
            o_gt, o_y = res["oc"]
            raw = words.tobytes()
            ints = [int.from_bytes(raw[32 * i:32 * i + 32], "little") * RINV % R for i in range(n * m)]  # out of Montgomery form
            x = pow(z, m, R)
            t_oo = timed(lambda: res.__setitem__("oo", old_open(ctx, kind, first, m, second, n, srs_g2, ints, o_y, x, z)),
                         a.old_reps)
            same = (o_gt.tolist() == codec.gt_enc(com).tolist() and np.array_equal(o_y.download((n, 24)), y_dev.download((n, 24)))
                    and res["oo"] == proof)
            emit({"what": "old", "kind": kname, "log_coeffs": lg, "commit_ms": t_oc, "open_ms": t_oo, "same_bytes": bool(same),
                  "commit_ratio": t_oc / t_commit, "open_ratio": t_oo / t_open})
            assert same, "old and new compositions differ"

            from torch.profiler import ProfilerActivity, profile

            for what, fn in (("commit", lambda: U.commit_dev(key, c, n * m, ctx)),
                             ("open", lambda: U.open_dev(key, c, n * m, y_dev, z, ctx))):
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    fn()
                    torch.cuda.synchronize()
                split = {s: 0.0 for s in KINDS}
                split["other"] = 0.0
                for e in prof.events():
                    if e.device_type != torch.autograd.DeviceType.CUDA:
                        continue
                    ms = (e.device_time if hasattr(e, "device_time") else e.cuda_time) / 1e3
                    k = next((s for s, keys in KINDS.items() if any(t in e.name for t in keys)), "other")
                    split[k] += ms
                emit({"what": "split", "call": what, "kind": kname, "log_coeffs": lg, **{s + "_ms": v for s, v in split.items()},
                      "kernels_ms": sum(split.values())})
            c.free()
    ctx.close()


if __name__ == "__main__":
    main()
