#!/usr/bin/env python3
"""bench.py -- RIPP inner-pairing-product hot path on B200 (contract: see the task statement).

Headline workload (BASELINE.json `metric`, configs[3]): TIPP aggregation of 2^12 Groth16 proofs on
BLS12-381 -- `aggregate_proofs` (ip_proofs/src/applications/groth16_aggregation.rs:77-160) on
trapdoor-simulated proofs and a powers-of-tau SRS (SURVEY.md §8d).  One step = one aggregation:
5 multi-pairings of 2^12 pairs, two device-resident GIPA recursions (12 rounds each), three KZG
opening MSMs, Fiat-Shamir hashing on the host.  Metric: prove seconds (lower is better).

  value        device-resident inputs, CUDA events on the library's stream, L2 flushed between steps
  e2e          the same aggregation through the host-pointer C-ABI call (ripp_tipp_aggregate): Groth16
               proofs in pinned host memory, H2D + kernels + D2H of the proof bytes, wall clock
  sub_metrics  verify_aggregate_proof of the emitted proof on the GPU (must accept), and
               the two leaf throughputs the metric string also names, measured in the same run:
               multi-Miller pairs/s (configs[1], 2^16 pairs per GPU) and G1 MSM points/s (configs[2] leaf,
               2^18 points per GPU), sharded by input slices with an NCCL all-gather of the per-rank
               partials when N > 1; and GIPA prove of ONE 2^18-element multiexponentiation instance
               (configs[2]) partitioned cyclically over the N ranks (strong scaling, same proof bytes at every N)
  roofline     integer-pipe (IMAD.WIDE) roofline of the dominant kernel class of the step, plus the
               Miller kernel at 2^16; peak = ripp_bench_imad measured live in this run
  cpu_baseline the compiled CPU restatement of the reference path (oracle/cpu, OpenMP on all host
               cores) running the same 2^12 aggregation once

N > 1 (weak scaling): every rank aggregates its own batch of 2^12 proofs; `value` is the max over
ranks of seconds per aggregation and `proofs_per_s` the whole-job rate.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Algorithmic Fq-product counts of the reference algorithm, measured by tests/test_hostsim.py::test_op_counts
# (own Fq12 accumulator per pair); one Fq Montgomery product = 2*12^2 + 12 = 300 MAC32 (SURVEY.md §8d).
FQ_MUL_PER_MILLER_PAIR = 6700
FQ_MUL_PER_FINAL_EXP = 7668   # + one Fq inversion, which is divsteps (modinv.cuh), not field products
FQ_MUL_PER_G1_MUL_255 = 255 * 7 + 127 * 11 + 4        # dbl-2009-l 2M+5S, madd-2007-bl 7M+4S, + to-affine products
FQ_MUL_PER_G2_MUL_128 = (128 * 16 + 64 * 29 + 10)     # same formulas over Fq2 (M2 = 3, S2 = 2 Fq products)
# SURVEY.md §8d (frozen): arkworks-style Pippenger, c = 16 -> 16 windows x one mixed Jacobian addition (11 Fq products)
# per point, bucket reduction not counted.  (Round 1 used 26 x 11 for its own c = 10 plan, which flattered the fraction.)
FQ_MUL_PER_G1_MSM_POINT = 16 * 11
MAC32_PER_FQ_MUL = 300
LOG_PROOFS = 12
LOG_PAIRS = 16
LOG_MSM = 18
LOG_GIPA = 18
# kernel class -> (kernel named in the line, ncu capture of that kernel under profiles/: `ncu --set full ... --page raw --csv`)
# timing categories of the library (include/ripp_b200.h: ripp_ctx_timing).  "msm" is the bucket accumulation -- the MSM's
# algorithmic work; its digit recoding / sort and its reduction + Horner tail are kernels of their own kind.
CLASS_KERNEL = {
    "msm_sort": ("k_msm_endo_expand / prepare / scan / scatter / size sort", "msm_sort"),
    "msm_reduce": ("k_msm_bucket_reduce + k_msm_window_sum + k_msm_horner_xt (bucket reduction and Horner tail)", "msm_reduce"),
    "fold": ("k_fold4_xp / k_fold4_xt (the four folds of a round in one launch: A' = A_R c + A_L, ..., gipa.rs:261-291) / k_fold_endo", "fold"),
    # the class's most frequent launch in the 2^12 aggregation is k_miller18<1> (18 of 26): its capture gives `traffic`;
    # the throughput kernel k_miller6<4,4> at 2^16 pairs has its own capture under roofline["miller_2^16"]
    "miller": ("k_miller18 / k_miller6 + Fq12 product tree (cfg_multi_pairing, inner_products/src/lib.rs:77-116)", "miller18"),
    "final_exp": ("k_final_exp18", "fexp"),
    "msm": ("k_msm_accumulate + fat-bucket kernels (bucket accumulation of the variable-base MSM)", "msm_acc"),
    "scale": ("k_scale_parts + k_scale_combine (a_i r^i, ck_i r^-i: groth16_aggregation.rs:118-131)", "scale"),
}
_UNIT = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}


def ncu_traffic(capture):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch (mean over the captured launches) from the newest committed
    `profiles/*_ncu_<capture>_raw.csv`; (None, None) when no capture of that kernel is committed."""
    import csv
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_%s_raw.csv" % capture)))
    if not files:
        return None, None
    try:
        rows = list(csv.reader(open(files[-1])))
        h = rows[0]
        ir, iw = h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum")
        vals = [float(r[ir]) * _UNIT[rows[1][ir]] + float(r[iw]) * _UNIT[rows[1][iw]] for r in rows[2:] if len(r) > max(ir, iw)]
        return (sum(vals) / len(vals) if vals else None), os.path.relpath(files[-1], ROOT)
    except Exception:
        return None, os.path.relpath(files[-1], ROOT)
METRIC = "tipp_groth16_aggregate_prove_seconds_at_2^12_proofs"
DTYPE = "u32-limb Montgomery (BLS12-381 Fq 381-bit / Fr 255-bit)"


_JSON_FD = None


def _claim_stdout():
    """stdout carries exactly the JSON line(s): anything a library prints to fd 1 (NCCL's version banner, whatever
    NCCL_DEBUG the box sets) is sent to stderr; the JSON is written to the saved descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit_json(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def _clock_sampler(stop, samples):
    q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    idx = os.environ.get("LOCAL_RANK", "0")
    while not stop.is_set():
        try:
            out = subprocess.run(["nvidia-smi", "-i", idx, "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=5).stdout.strip()
            if out:
                samples.append([x.strip() for x in out.split(",")])
        except Exception:
            pass
        stop.wait(0.2)


def _clocks_summary(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
    sm = sorted(int(s[0]) for s in samples if s[0].isdigit())
    reasons = set()
    for s in samples:
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
            if v.lower().startswith("active"):
                reasons.add(name)
    return {"sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": int(samples[0][1]) if samples[0][1].isdigit() else None, "reasons": sorted(reasons)}


def _host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def tipp_algorithmic_macs(n):
    """MAC32 per aggregation by kernel class (SURVEY.md App. C op inventory)."""
    lg = n.bit_length() - 1
    return {
        "miller": (13 * n - 8) * FQ_MUL_PER_MILLER_PAIR * MAC32_PER_FQ_MUL,
        "final_exp": (5 + 8 * lg) * FQ_MUL_PER_FINAL_EXP * MAC32_PER_FQ_MUL,
        "fold": (3 * (n - 1) * FQ_MUL_PER_G1_MUL_255 + 3 * (n - 1) * FQ_MUL_PER_G2_MUL_128) * MAC32_PER_FQ_MUL,
        "scale": (n * FQ_MUL_PER_G1_MUL_255 + n * 2 * FQ_MUL_PER_G2_MUL_128) * MAC32_PER_FQ_MUL,
        "msm": ((n + 2 * (n - 1) + (2 * n - 1)) * FQ_MUL_PER_G1_MSM_POINT + 2 * (2 * n - 1) * 3 * FQ_MUL_PER_G1_MSM_POINT) * MAC32_PER_FQ_MUL,
    }


def run_reference(args):
    """The reference's CPU path (compiled restatement, all host cores) on the same workload."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import cpu_baseline

    n = 1 << args.logn
    # all host cores, whatever OMP_NUM_THREADS says (torch.distributed.run exports OMP_NUM_THREADS=1 to every rank)
    work = cpu_baseline.TippWorkload(n, threads=_host_threads())
    work.run()  # one untimed warm-up: page in the tables, spin up the OpenMP team
    times = sorted(work.run() for _ in range(args.steps))
    v = times[len(times) // 2]  # median
    info = work.info()
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": 1, "ms_per_step": 1e3 * v, "higher_is_better": False, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": {"workload": "TIPP aggregate_proofs of 2^%d Groth16 proofs, BLS12-381 (BASELINE configs[3]); CPU restatement of the reference path" % args.logn,
                   "proofs": n},
        "cpu_baseline": {"value": v, "unit": "s", "cores": info["cores"], "kind": info["kind"], "sample": info["sample"]},
        "e2e": {"value": v, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "proofs_per_s": n / v,
    }
    print(json.dumps(line))


def run_config5(args):
    """BASELINE configs[4]: scaling sweep of the two leaf inner products.  Each point is ONE instance of n elements
    sharded by contiguous slices over the ranks through the library's own entry points (ripp_pairing_ip_sharded_dev /
    ripp_msm_g1_sharded_dev: per-rank partial, one ncclAllGather, combine on every rank).  CUDA events on the shared
    stream, max over ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from ripp_b200 import _lib, synth

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    _claim_stdout()
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = _lib.Context(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    if world > 1:
        from ripp_b200.parallel import init_library_comm

        init_library_comm(ctx)  # the sharded entry points run their all-gathers inside the library (comm.cu)
    imad_peak, _ = ctx.bench_imad(0, 4096)
    max_p, max_m = 20, 22

    def timed(fn, reps=3):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for s_, e_ in evs:
            s_.record()
            fn()
            e_.record()
        torch.cuda.synchronize()
        t = torch.tensor([min(s_.elapsed_time(e_) for s_, e_ in evs)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def emit(line):
        if rank == 0:
            _emit_json(line)

    nl_p = (1 << max_p) // world
    a = synth.g1_points_dev(ctx, "cfg5-a", nl_p, seed=rank)
    b = synth.g2_points_dev(ctx, "cfg5-b", nl_p, seed=rank)
    part = torch.zeros(144, dtype=torch.int32, device="cuda")
    gath = torch.zeros(world * 144, dtype=torch.int32, device="cuda")
    res = torch.zeros(144, dtype=torch.int32, device="cuda")
    for lg in range(10, max_p + 1, 2):
        n = 1 << lg
        nl = n // world

        def pairing():
            ctx.pairing_ip_sharded_dev(a, b, nl, res.data_ptr())

        ms = timed(pairing)
        emit({"config": "BASELINE configs[4]", "op": "PairingInnerProduct", "log_n": lg, "n_gpus": world, "scaling": "strong",
              "ms": round(ms, 3), "pairs_per_s": round(n / ms * 1e3),
              "frac_of_imad_wide_peak_all_gpus": round(n * FQ_MUL_PER_MILLER_PAIR * MAC32_PER_FQ_MUL / (ms * 1e-3) / (imad_peak * world), 4)})
    a.free()
    b.free()
    nl_m = (1 << max_m) // world
    bases = synth.g1_points_dev(ctx, "cfg5-m", nl_m, seed=rank)
    sc = ctx.to_device(synth.scalars_mont("cfg5-s", nl_m, seed=rank))
    ppt = torch.zeros(24, dtype=torch.int32, device="cuda")
    gpt = torch.zeros(world * 24, dtype=torch.int32, device="cuda")
    rpt = torch.zeros(24, dtype=torch.int32, device="cuda")
    for lg in range(10, max_m + 1, 2):
        n = 1 << lg
        nl = n // world

        def msm():
            ctx.msm_sharded_dev(1, bases, sc, nl, rpt.data_ptr())

        ms = timed(msm)
        emit({"config": "BASELINE configs[4]", "op": "MultiexponentiationInnerProduct<G1>", "log_n": lg, "n_gpus": world,
              "scaling": "strong", "ms": round(ms, 3), "points_per_s": round(n / ms * 1e3)})
    bases.free()
    sc.free()
    if world == 1:
        # the reference's CPU path beside it (compiled restatement, all host cores), bounded sizes
        from oracle import cpu_baseline

        for lg in (10, 14):
            r = cpu_baseline.pairing_pairs_per_s(1 << lg)
            emit({"config": "BASELINE configs[4]", "op": "PairingInnerProduct", "impl": "cpu restatement (port)", "log_n": lg,
                  "cores": r["cores"], "ms": round(1e3 * r["seconds"], 1), "pairs_per_s": round(r["value"])})
        for lg in (14, 18):
            r = cpu_baseline.msm_points_per_s(1 << lg)
            emit({"config": "BASELINE configs[4]", "op": "MultiexponentiationInnerProduct<G1>", "impl": "cpu restatement (port)",
                  "log_n": lg, "cores": r["cores"], "ms": round(1e3 * r["seconds"], 1), "points_per_s": round(r["value"])})
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--logn", type=int, default=LOG_PROOFS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub-metrics", action="store_true")
    ap.add_argument("--config5", action="store_true",
                    help="BASELINE configs[4] instead of the headline: sweep n = 2^10 .. 2^22 of the pairing and MSM inner "
                         "products, ONE instance of n elements sharded over the N ranks (strong scaling), one JSON line per point; "
                         "at N = 1 the CPU restatement is timed beside it on bounded sizes")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy: "
                         "aggregate_proof.npy = the AggregateProof bytes, one float32 per byte.  The inputs are seeded, so two "
                         "builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config5):
        ap.error("--dump-outputs applies to the headline GPU workload only")
    if args.impl == "reference":
        return run_reference(args)
    if args.config5:
        return run_config5(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from ripp_b200 import _lib, codec, synth

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    # rank 0 prints exactly ONE JSON line on stdout: NCCL's version banner (it goes to fd 1 whenever NCCL_DEBUG is
    # set, whatever NCCL_DEBUG_FILE says) is diverted to stderr
    _claim_stdout()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = _lib.Context(local_rank)
    # one non-default stream shared by torch (events, NCCL ordering) and the library's kernels
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    if world > 1:
        # the library's own NCCL communicator (comm.cu): the sharded entry points run their all-gathers inside the C ABI
        from ripp_b200.parallel import init_library_comm

        init_library_comm(ctx)
    warmup = max(args.warmup, 3)
    n = 1 << args.logn

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    # ---- headline: TIPP aggregation, this rank's batch of 2^12 proofs generated on the GPU -------
    inst = synth.tipp_instance_dev(ctx, n, seed=rank)

    def step():
        return ctx.tipp_aggregate_dev(inst["srs_g1"], inst["srs_g2"], inst["a"], inst["b"], inst["c"], n)

    for _ in range(warmup):
        proof = step()
    barrier()
    stop, samples = threading.Event(), []
    th = threading.Thread(target=_clock_sampler, args=(stop, samples), daemon=True)
    th.start()

    launches0 = ctx.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for s, e in ev:
        flush.zero_()
        s.record()
        proof = step()
        e.record()
    barrier()
    launches = ctx.launches - launches0
    ms_total = max_over_ranks(sum(s.elapsed_time(e) for s, e in ev))
    value_s = ms_total / args.steps / 1e3
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "aggregate_proof.npy"), np.frombuffer(proof, dtype=np.uint8).astype(np.float32))

    # per-class device time of one aggregation (instrumented pass, outside the timed region)
    ctx.set_timing(True)
    ctx.timing()
    step()
    breakdown = ctx.timing()
    ctx.set_timing(False)

    # ---- end to end through the host-pointer C ABI ------------------------------------------------
    a_h = torch.from_numpy(inst["a"].download((n, 24)).view(np.int32)).pin_memory()
    b_h = torch.from_numpy(inst["b"].download((n, 48)).view(np.int32)).pin_memory()
    c_h = torch.from_numpy(inst["c"].download((n, 24)).view(np.int32)).pin_memory()
    a_np, b_np, c_np = (t.numpy().view(np.uint32) for t in (a_h, b_h, c_h))
    host_proof = ctx.tipp_aggregate(inst["srs_g1"], inst["srs_g2"], a_np, b_np, c_np)
    assert host_proof == proof, "host-pointer and device-resident entry points disagree"
    e2e_steps = max(2, min(args.steps, 5))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        host_proof = ctx.tipp_aggregate(inst["srs_g1"], inst["srs_g2"], a_np, b_np, c_np)
    e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)

    # ---- the verifier of the same statement on the GPU (groth16_aggregation.rs:162-231) -------------
    sub = {}
    assert ctx.tipp_verify_aggregate(inst["vsrs"], inst["vk"], inst["inputs"], host_proof), "aggregate proof rejected"
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ctx.tipp_verify_aggregate(inst["vsrs"], inst["vk"], inst["inputs"], host_proof)
    sub["verify_aggregate_s"] = {"value": max_over_ranks((time.perf_counter() - t0) / e2e_steps), "proofs_per_gpu": n,
                                 "accepted": True, "timing": "wall clock through the host-pointer C ABI"}

    # ---- leaf throughputs (sharded by input slices; one partial per rank all-gathered) -------------
    miller_k_ms = None
    if not args.no_sub_metrics:
        npairs = 1 << LOG_PAIRS
        pa = synth.g1_points_dev(ctx, "cfg2-m", npairs, seed=rank)
        pb = synth.g2_points_dev(ctx, "cfg2-k", npairs, seed=rank)
        partial = torch.zeros(144, dtype=torch.int32, device="cuda")
        gathered = torch.zeros(world * 144, dtype=torch.int32, device="cuda")
        result = torch.zeros(144, dtype=torch.int32, device="cuda")

        def pairing_step():
            # world == 1: the plain entry point; else Miller partial -> ncclAllGather (576 B / rank) -> product + final exp
            ctx.pairing_ip_sharded_dev(pa, pb, npairs, result.data_ptr())

        def timed(fn, reps):
            for _ in range(3):
                fn()
            barrier()
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for s, e in evs:
                flush.zero_()
                s.record()
                fn()
                e.record()
            barrier()
            return max_over_ranks(sum(s.elapsed_time(e) for s, e in evs)) / reps

        reps = max(3, min(args.steps, 5))
        ms = timed(pairing_step, reps)
        miller_k_ms = timed(lambda: ctx.miller_partial_dev(pa, pb, npairs, partial.data_ptr()), reps)
        sub["miller_pairs_per_s"] = {"value": world * npairs / (ms * 1e-3), "pairs_per_gpu": npairs, "ms_per_step": ms,
                                     "miller_kernel_ms": miller_k_ms}
        pa.free()
        pb.free()
        nmsm = 1 << LOG_MSM
        bases = synth.g1_points_dev(ctx, "cfg3-a", nmsm, seed=rank)
        sc = ctx.to_device(synth.scalars_mont("cfg3-b", nmsm, seed=rank))
        part_pt = torch.zeros(24, dtype=torch.int32, device="cuda")
        gath_pt = torch.zeros(world * 24, dtype=torch.int32, device="cuda")
        ones = ctx.to_device(codec.fr_vec_enc([1] * world))
        res_pt = torch.zeros(24, dtype=torch.int32, device="cuda")

        def msm_step():
            ctx.msm_sharded_dev(1, bases, sc, nmsm, res_pt.data_ptr())

        ms = timed(msm_step, reps)
        sub["msm_g1_points_per_s"] = {"value": world * nmsm / (ms * 1e-3), "points_per_gpu": nmsm, "ms_per_step": ms}
        bases.free()
        sc.free()

        # ---- BASELINE configs[2] (ii): GIPA prove, multiexponentiation instantiation (benches/benches/gipa.rs:86-94),
        # ONE global instance of 2^18 elements partitioned cyclically over the ranks (strong scaling: the same proof
        # bytes at every N; parallel.py).  Wall clock, max over ranks: the round loop includes the host's hashing.
        import hashlib

        from ripp_b200.parallel import Comm, ShardedGIPA

        ng = 1 << LOG_GIPA
        nl = ng // world

        def share(tag, group):
            sc_h = synth.scalars_mont(tag, ng)[rank::world]
            if group == 0:
                return torch.from_numpy(np.ascontiguousarray(sc_h).view(np.int32)).cuda()
            d = ctx.to_device(np.ascontiguousarray(sc_h))
            t = torch.empty((nl, 24 if group == 1 else 48), dtype=torch.int32, device="cuda")
            (ctx.g1_scale_dev if group == 1 else ctx.g2_scale_dev)(None, d, nl, t.data_ptr())
            ctx.sync()
            d.free()
            return t

        ga, gb, gv, gw = share("cfg3-a", 1), share("cfg3-b", 0), share("cfg3-v", 2), share("cfg3-w", 1)

        def gipa_step():
            # ripp_gipa_prove_sharded_dev: the round loop, its all-gathers (NCCL inside the library) and the resident tail
            return ctx.gipa_prove_sharded_dev(_lib.GIPA_MULTIEXP_PEDERSEN, ga.data_ptr(), gb.data_ptr(), gv.data_ptr(),
                                              gw.data_ptr(), nl, world)[0]

        gproof = gipa_step()  # warm-up
        g_reps = 2
        barrier()
        t0 = time.perf_counter()
        for _ in range(g_reps):
            gproof = gipa_step()
        torch.cuda.synchronize()
        g_s = max_over_ranks((time.perf_counter() - t0) / g_reps)
        sub["gipa_multiexp_prove_s"] = {"value": g_s, "elements_total": ng, "elements_per_gpu": nl, "scaling": "strong",
                                        "proof_blake2b": hashlib.blake2b(gproof, digest_size=16).hexdigest(),
                                        "proof_bytes": len(gproof)}
        del ga, gb, gv, gw

        # ---- strong scaling of ONE instance over the N ranks (SURVEY.md §8e), all through the library's sharded entry
        # points: leaf products at sizes where a GPU is past its latency floor, and one batch of 2^16 proofs
        def rand_fr(count, seed):
            w = np.random.default_rng(seed).integers(0, 1 << 32, size=(count, 8), dtype=np.uint32)
            w[:, 7] &= 0x0FFFFFFF  # < r: a valid Montgomery representative
            return w

        def gen(group, count, seed):
            e = ctx.to_device(rand_fr(count, seed))
            out = ctx.alloc(count * (96 if group == 1 else 192))
            ctx.fixed_base_msm_dev(group, None, e, count, out)
            ctx.sync()
            e.free()
            return out

        strong = {}
        lp, lm, la = 18, 22, 16
        nlp = (1 << lp) // world
        spa, spb = gen(1, nlp, 1000 + rank), gen(2, nlp, 2000 + rank)
        ms = timed(lambda: ctx.pairing_ip_sharded_dev(spa, spb, nlp, result.data_ptr()), 3)
        strong["pairing_ip_2^%d" % lp] = {"ms": ms, "pairs_per_s": (1 << lp) / (ms * 1e-3)}
        spa.free()
        spb.free()
        nlm = (1 << lm) // world
        smb, sms = gen(1, nlm, 3000 + rank), ctx.to_device(rand_fr(nlm, 4000 + rank))
        ms = timed(lambda: ctx.msm_sharded_dev(1, smb, sms, nlm, res_pt.data_ptr()), 3)
        strong["msm_g1_2^%d" % lm] = {"ms": ms, "points_per_s": (1 << lm) / (ms * 1e-3)}
        smb.free()
        sms.free()
        strong["gipa_multiexp_2^%d" % LOG_GIPA] = {"s": g_s}
        na = 1 << la
        big = synth.tipp_instance_dev(ctx, na, seed=7)

        def cyc(buf, words):
            return ctx.to_device(np.ascontiguousarray(buf.download((na, words))[rank::world]))

        if world == 1:
            agg_step = lambda: ctx.tipp_aggregate_dev(big["srs_g1"], big["srs_g2"], big["a"], big["b"], big["c"], na)
        else:
            ca, cb, cc = cyc(big["a"], 24), cyc(big["b"], 48), cyc(big["c"], 24)
            agg_step = lambda: ctx.tipp_aggregate_sharded_dev(big["srs_g1"], big["srs_g2"], ca, cb, cc, na)
        aproof = agg_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            aproof = agg_step()
        a_s = max_over_ranks((time.perf_counter() - t0) / 2)
        strong["tipp_aggregate_2^%d" % la] = {"s": a_s, "proof_blake2b": hashlib.blake2b(aproof, digest_size=16).hexdigest()}
        sub["strong_scaling_one_instance"] = strong
        del big

    stop.set()
    th.join(timeout=2)

    # ---- roofline ----------------------------------------------------------------------------------
    imad_peak, _ = ctx.bench_imad(0, 4096)
    imad32_peak, _ = ctx.bench_imad(1, 4096)
    chain_peak, _ = ctx.bench_imad(2, 4096)
    macs = tipp_algorithmic_macs(n)
    # dominant kernel group = largest summed device time among ALL accounted groups; the MSM's algorithmic MAC32 are
    # credited to the whole MSM (sort + accumulate + reduce) in step_frac_by_class and to none of its overhead groups alone
    groups = [c for c in breakdown if c != "other"]
    dom = max(groups, key=lambda c: breakdown[c][0])
    dom_ms, dom_launches = breakdown[dom]
    msm_ms = sum(breakdown[c][0] for c in ("msm", "msm_sort", "msm_reduce") if c in breakdown)
    dom_macs = macs.get(dom, 0.0) if dom in ("miller", "final_exp", "fold", "scale") else (macs["msm"] if dom == "msm" else 0.0)
    achieved = dom_macs / (dom_ms * 1e-3) if dom_ms else 0.0
    traffic, traffic_src = ncu_traffic(CLASS_KERNEL[dom][1])
    all_ms = sum(breakdown[c][0] for c in breakdown)
    roofline = {
        "bound": "int32 multiply pipe (IMAD.WIDE.U32: one 32x32+64 MAC per lane-instruction)",
        # the kernel class with the largest summed device time in one aggregation (CUDA events around every launch of
        # the class, on the launching stream; classes overlap on several streams, so the sum over classes exceeds the step)
        "kernel": CLASS_KERNEL[dom][0], "launches": dom_launches, "mean_ms": dom_ms / max(dom_launches, 1),
        "share_of_summed_kernel_time": dom_ms / all_ms if all_ms else None,
        "achieved": achieved / 1e12, "peak": imad_peak / 1e12, "unit": "TMAC32/s", "frac": achieved / imad_peak,
        "traffic": traffic, "traffic_source": traffic_src,
        "note": ("2^12 proofs is a latency regime: most of these %d launches are a few CTAs each (one dependent chain per pair "
                 "below 1184 pairs), so the fraction of the whole-GPU integer peak is small by construction; the throughput "
                 "kernels the north star names are reported at their own sizes in miller_2^16 / msm_2^18" % dom_launches),
        "peak_source": "ripp_bench_imad in this run: independent IMAD.WIDE.U32 chains, all SMs",
        "peak_imad32_tmacs": imad32_peak / 1e12, "peak_carry_chain_tmacs": chain_peak / 1e12,
        "step_breakdown_ms": {c: round(breakdown[c][0], 3) for c in breakdown},
        "step_launches": {c: breakdown[c][1] for c in breakdown},
        "step_frac_by_class": {c: (macs[c] / ((msm_ms if c == "msm" else breakdown[c][0]) * 1e-3) / imad_peak
                                   if (msm_ms if c == "msm" else breakdown[c][0]) else None) for c in macs},
        "whole_step_frac": sum(macs.values()) / value_s / imad_peak,
    }
    if miller_k_ms:
        m = (1 << LOG_PAIRS) * FQ_MUL_PER_MILLER_PAIR * MAC32_PER_FQ_MUL / (miller_k_ms * 1e-3)
        roofline["miller_2^16"] = {"kernel": "k_miller6<4,4> + Fq12 product tree", "kernel_ms": miller_k_ms,
                                   "traffic": ncu_traffic("miller6")[0],
                                   "achieved": m / 1e12, "frac": m / imad_peak,
                                   "mac32_per_pair": FQ_MUL_PER_MILLER_PAIR * MAC32_PER_FQ_MUL}

    if "msm_g1_points_per_s" in sub:
        mm = sub["msm_g1_points_per_s"]
        m = world * mm["points_per_gpu"] * FQ_MUL_PER_G1_MSM_POINT * MAC32_PER_FQ_MUL / (mm["ms_per_step"] * 1e-3) / world
        roofline["msm_2^18"] = {"kernel": "whole G1 MSM (expand, prepare, scan, scatter, accumulate, fat buckets, reductions, Horner)",
                                "traffic_accumulate_kernel": ncu_traffic("msm_acc")[0],
                                "kernel_ms": mm["ms_per_step"], "achieved": m / 1e12, "frac": m / imad_peak,
                                "mac32_per_point": FQ_MUL_PER_G1_MSM_POINT * MAC32_PER_FQ_MUL}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value_s, "unit": "s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": "TIPP aggregate_proofs of 2^%d Groth16 proofs per GPU, BLS12-381, Blake2b (BASELINE configs[3])" % args.logn,
                       "proofs_per_gpu": n, "l2": "flushed between steps (256 MiB memset)",
                       "parallelism": "one 2^%d-proof aggregation per GPU (weak); strong_scaling: ONE instance sharded over the N ranks "
                                      "through the library's NCCL entry points (same bytes at every N)" % args.logn,
                       "strong_scaling": sub.get("strong_scaling_one_instance")},
            "proofs_per_s": world * n / value_s,
            "e2e": {"value": e2e_s, "unit": "s", "h2d_bytes_per_step": n * 384, "d2h_bytes_per_step": len(host_proof)},
            "gpu_launches": launches,
            "clocks": _clocks_summary(samples),
            "roofline": roofline,
            "sub_metrics": sub,
        }
        if not args.no_cpu_baseline and world == 1:
            try:
                from oracle import cpu_baseline

                work = cpu_baseline.TippWorkload(n, threads=_host_threads())
                work.run()  # warm-up
                secs = sorted(work.run() for _ in range(3))[1]
                info = work.info()
                line["cpu_baseline"] = {"value": secs, "unit": "s", "cores": info["cores"], "kind": info["kind"],
                                        "sample": info["sample"] + "; median of 3 after one warm-up"}
                # the checker's proof of the same seeded statement, byte for byte against the GPU's (the oracle is the
                # checker here, never the thing measured)
                from oracle import protocols as O

                line["parity_bytes_equal"] = bool(O.ser_aggregate_proof(work.proof) == proof == host_proof)
                line["parity_note"] = ("AggregateProof bytes (%d B) of the timed GPU step == the CPU oracle's proof of the same "
                                       "synthetic instance (seed 0)" % len(proof))
            except Exception as ex:  # the GPU numbers stand on their own
                line["cpu_baseline"] = {"value": None, "unit": "s", "cores": 0, "kind": "port", "sample": "failed: %r" % (ex,)}
        _emit_json(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
