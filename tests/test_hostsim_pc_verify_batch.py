"""The final-key exponent rule of the batched polynomial-commitment verifier (ripp_b200/csrc/pc_scan.cuh
pc::key_exponent, the index rule of k_pc_key_exponents_seg) compiled for the host: exponent i of instance k is
prod over the bits j set in i of t_{k,j}^-1, optionally times a per-instance factor.  Compared with the order of the
oracle's GIPA.compute_final_commitment_keys (gipa.rs:365-399), and the key it builds from them with the oracle's key."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import poly_commit as OPC
from oracle import synth as OS
from ripp_b200 import codec as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hs():
    src = os.path.join(ROOT, "tests", "hostsim", "hostsim_pc_verify_batch.cpp")
    so = os.path.join(ROOT, "tests", "hostsim", "_hostsim_pc_verify_batch.so")
    csrc = os.path.join(ROOT, "ripp_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".h"))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _enc(vals):
    return C.fr_vec_enc(vals) if vals else np.zeros((1, 8), dtype=np.uint32)


def _exponents(hs, transcripts, L, factors=None):
    count = len(transcripts)
    tinv = np.ascontiguousarray(_enc([E.fr_inv(c) for t in transcripts for c in t]))
    fac = np.ascontiguousarray(_enc(factors)) if factors is not None else None
    out = np.zeros((count << L, 8), dtype=np.uint32)
    hs.hs_key_exponents(_ptr(tinv), ctypes.c_uint(L), _ptr(fac) if fac is not None else None, ctypes.c_size_t(count), _ptr(out))
    return [[C.fr_dec(w) for w in out[k << L:(k + 1) << L]] for k in range(count)]


def _final_key_exponents(transcript):
    """The exponents of ck_a in the order GIPA.compute_final_commitment_keys (oracle/protocols.py) applies them."""
    ea = [1]
    for i, c in enumerate(transcript):
        c_inv = E.fr_inv(c)
        for j in range(2 ** i):
            ea.append(ea[j] * c_inv % E.R)
    return ea


@pytest.mark.parametrize("count,L", [(1, 0), (1, 1), (3, 4), (2, 7), (5, 3)])
def test_key_exponents_match_final_key_order(hs, count, L):
    rnd = random.Random(31 * count + L)
    transcripts = [[rnd.randrange(1, E.R) for _ in range(L)] for _ in range(count)]
    factors = [rnd.randrange(E.R) for _ in range(count)]
    factors[0] = 0
    plain, scaled = _exponents(hs, transcripts, L), _exponents(hs, transcripts, L, factors)
    for k in range(count):
        want = _final_key_exponents(transcripts[k])
        assert plain[k] == want, (count, L, k)
        assert scaled[k] == [e * factors[k] % E.R for e in want], (count, L, k)


@pytest.mark.parametrize("L", [1, 3])
def test_key_from_exponents_is_the_oracle_final_key(hs, L):
    """sum_i e_i w_i over a first-tier key equals the key the oracle's SCALAR_SSM_G1 verifier folds to."""
    rnd = random.Random(L)
    transcript = [rnd.randrange(1, E.R) for _ in range(L)]
    key = OS.g1_points("hs-pcv-key", 1 << L)
    gipa = OPC._first_tier().gipa
    want, _ = gipa.compute_final_commitment_keys((key, [None] * len(key), None), transcript)
    got = E.msm(key, _exponents(hs, [transcript], L)[0], E.g1_add, E.g1_mul)
    assert got == want
