"""Timing of validated proof ingestion: decoding ark-groth16 Proof records (A, B, C as ark-serialize bytes) on the GPU,
against the CPU restatement of the same rules, and aggregate_proofs from the bytes against aggregate_proofs from
Montgomery limbs.  One JSON line per size (default 2^12 and 2^16 proofs):

  gpu_decode_ms          {compressed, uncompressed}: device-event time of the three decode launches (A, B, C of every
                         record, records resident on the device), median of --reps
  cpu_restatement_ms     {compressed, uncompressed}: oracle/cpu/serde_cpu.cpp's decode of the same records on all host cores (OpenMP) --
                         CPU restatement (not arkworks), as bench.py labels its CPU arm
  aggregate_ms           (2^12 only) host clock around ripp_tipp_aggregate_serialized (compressed records in host memory)
                         and around ripp_tipp_aggregate (the same points as Montgomery limbs), alternated, median; with
                         proof_bytes_equal
  device, power_limit_w  read in the same call

Usage: python tools/time_deserialize.py [--log2 12 16] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from oracle import serde_cases as SC  # noqa: E402
from oracle.cpu import serde_binding as SB  # noqa: E402
from ripp_b200 import _lib, synth  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out)
    except Exception:
        power = None
    return name, power


def gpu_decode_ms(ctx, data, n, compressed, reps):
    g1b = 48 if compressed else 96
    rec = 4 * g1b
    buf = ctx.to_device(np.frombuffer(data, dtype=np.uint8).copy())
    a, b, c = ctx.alloc(n * 96), ctx.alloc(n * 192), ctx.alloc(n * 96)
    st = ctx.alloc(3 * n)
    stream = torch.cuda.ExternalStream(ctx.stream)  # events on the library's own stream
    ms = []
    for r in range(reps + 1):  # the first pass loads the module
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.g1_deserialize_dev(buf.ptr, n, rec, compressed, a, st.ptr)
        ctx.g2_deserialize_dev(buf.ptr + g1b, n, rec, compressed, b, st.ptr + n)
        ctx.g1_deserialize_dev(buf.ptr + 3 * g1b, n, rec, compressed, c, st.ptr + 2 * n)
        e1.record(stream)
        e1.synchronize()
        if r:
            ms.append(e0.elapsed_time(e1))
    status = st.download(3 * n, dtype=np.uint8)
    assert not status.any(), "valid records were rejected"
    return float(np.median(ms))


def cpu_decode_ms(data, n, compressed, reps):
    g1b = 48 if compressed else 96
    rec = 4 * g1b
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        for group, off in ((1, 0), (2, g1b), (1, 3 * g1b)):
            _, st = SB.deserialize(group, data[off:], n, rec, compressed)
            assert not st.any()
        ms.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2", type=int, nargs="+", default=[12, 16])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cpu-reps", type=int, default=2)
    args = ap.parse_args()
    ctx = _lib.Context(0)
    cpu_threads = SB.threads()
    name, power = card()
    for lg in args.log2:
        n = 1 << lg
        if lg == 12:
            inst = synth.tipp_instance_dev(ctx, n)
            pa, pb, pc = inst["a"], inst["b"], inst["c"]
        else:
            pa, pb, pc = synth.g1_points_dev(ctx, "serde-a", n), synth.g2_points_dev(ctx, "serde-b", n), synth.g1_points_dev(ctx, "serde-c", n)
        a_h, b_h, c_h = pa.download((n, 24)), pb.download((n, 48)), pc.download((n, 24))
        line = {"n_proofs": n, "device": name, "power_limit_w": power, "gpu_decode_ms": {}, "cpu_restatement_ms": {},
                "cpu_restatement_label": "CPU restatement (not arkworks), %d threads" % cpu_threads}
        records = {}
        for compressed in (True, False):
            key = "compressed" if compressed else "uncompressed"
            records[key] = SC.proof_records(a_h, b_h, c_h, compressed)
            line["gpu_decode_ms"][key] = round(gpu_decode_ms(ctx, records[key], n, compressed, args.reps), 3)
            line["cpu_restatement_ms"][key] = round(cpu_decode_ms(records[key], n, compressed, args.cpu_reps), 1)
        if lg == 12:
            s1, s2 = inst["srs_g1"], inst["srs_g2"]
            t_ser, t_limbs = [], []
            got = want = None
            for r in range(args.reps + 1):
                t0 = time.perf_counter()
                got = ctx.tipp_aggregate_serialized(s1, s2, records["compressed"], n, True)
                t1 = time.perf_counter()
                want = ctx.tipp_aggregate(s1, s2, a_h, b_h, c_h)
                t2 = time.perf_counter()
                if r:
                    t_ser.append(1e3 * (t1 - t0))
                    t_limbs.append(1e3 * (t2 - t1))
            agg = float(np.median(t_limbs))
            line["aggregate_ms"] = {"serialized_compressed": round(float(np.median(t_ser)), 2), "montgomery_limbs": round(agg, 2),
                                    "proof_bytes_equal": got == want}
            line["gpu_decode_share_of_aggregate"] = {k: round(v / agg, 4) for k, v in line["gpu_decode_ms"].items()}
        print(json.dumps(line), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
