"""The scalar rules of Groth16 verification by random linear combination (ripp_b200/csrc/rlc.cuh and hash.h's
ChaCha20 block, run by k_rlc_scalars and k_rlc_segment_fr) compiled for the host against the oracle
(oracle/groth16_rlc.py)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import encoding as enc
from oracle import groth16_rlc as Q
from ripp_b200 import codec as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hs():
    src = os.path.join(ROOT, "tests", "hostsim", "hostsim_rlc.cpp")
    so = os.path.join(ROOT, "tests", "hostsim", "_hostsim_rlc.so")
    csrc = os.path.join(ROOT, "ripp_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".h"))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


@pytest.mark.parametrize("seed", [bytes(32), bytes(range(32)), bytes(range(255, 223, -1))], ids=["zero", "up", "down"])
def test_block_and_scalars_match_oracle(hs, seed):
    key = np.frombuffer(seed, dtype=np.uint8).copy()
    members = [True] * (4 * 9 + 1)  # the last one is normalised; blocks 0..8 stay raw
    want = Q.rlc_scalars(seed, members, len(members) + 1)
    for b in (0, 1, 2, 8):
        blk = np.zeros(64, dtype=np.uint8)
        hs.hs_chacha20_block(_ptr(key), ctypes.c_uint64(b), _ptr(blk))
        assert blk.tobytes() == enc.chacha20_block(seed, b), b
        out = np.zeros(32, dtype=np.uint32)
        hs.hs_rlc_scalars4(_ptr(key), ctypes.c_uint64(b), _ptr(out))
        assert [C.fr_dec(out[8 * q : 8 * q + 8]) for q in range(4)] == want[4 * b : 4 * b + 4], b
    # a block counter above 2^32 (the 64-bit counter of rand_chacha's layout)
    blk = np.zeros(64, dtype=np.uint8)
    hs.hs_chacha20_block(_ptr(key), ctypes.c_uint64((1 << 32) + 5), _ptr(blk))
    assert blk.tobytes() == enc.chacha20_block(seed, (1 << 32) + 5)


@pytest.mark.parametrize("k", [1, 2, 7, 58])
def test_normalisation_matches_oracle(hs, k):
    seed = bytes(range(32))
    r = Q.rlc_scalars(seed, [True] * k, k)
    raw = Q.rlc_scalars(seed, [True] * k, k + 1)  # the ChaCha values before normalisation
    words = np.concatenate([C.fr_enc(v) for v in raw]).astype(np.uint32)
    out = np.zeros(8, dtype=np.uint32)
    hs.hs_rlc_last(_ptr(words), ctypes.c_uint32(k), _ptr(out))
    assert C.fr_dec(out) == r[-1]
    assert (sum(raw[:-1]) + C.fr_dec(out)) % E.R == 1
