"""The public-input rule of the Groth16 kernels (serde::decode_fr in ripp_b200/csrc/serde.cuh, run by
k_fr_deserialize) compiled for the host against the oracle: canonical iff < r, Montgomery form, zero when rejected."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import groth16 as G
from ripp_b200 import codec as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hs():
    src = os.path.join(ROOT, "tests", "hostsim", "hostsim_groth16.cpp")
    so = os.path.join(ROOT, "tests", "hostsim", "_hostsim_groth16.so")
    csrc = os.path.join(ROOT, "ripp_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def test_fr_decode_matches_oracle(hs):
    rng = random.Random(5)
    vals = [0, 1, 2, E.R - 1, E.R, E.R + 1, (1 << 255) - 1, 1 << 255, (1 << 256) - 1]
    vals += [rng.randrange(E.R) for _ in range(64)] + [rng.randrange(E.R, 1 << 256) for _ in range(64)]
    for v in vals:
        data = v.to_bytes(32, "little")
        (want,), canonical = G.decode_inputs(data, 1)
        out = np.zeros(8, dtype=np.uint32)
        buf = np.frombuffer(data, dtype=np.uint8).copy()
        ok = hs.hs_fr_decode(ctypes.c_void_p(buf.ctypes.data), ctypes.c_void_p(out.ctypes.data))
        assert bool(ok) == canonical == (v < E.R), hex(v)
        assert np.array_equal(out, C.fr_enc(want) if canonical else np.zeros(8, dtype=np.uint32)), hex(v)
