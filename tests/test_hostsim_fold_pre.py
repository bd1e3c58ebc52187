"""The fold over precomputed bases (k_fold_pre + k_fold4_xp<true>): endo.cuh's split recoding -- every endomorphism
digit's NAF cut at bit H, the high digits moved onto D = [2^H] P -- and xt.cuh's team formulas, compiled for the host
(emulated carry flag, as tests/test_hostsim.py does), against the Python oracle's k P + lo."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import bls12_381 as E
from ripp_b200 import codec as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
rnd = random.Random(20261020)
LAM = E.X_ABS**2 - 1
H = {1: 64, 2: 32}
BASE = {1: LAM, 2: E.X_ABS}  # eigenvalue of E on the group: phi = [lambda] on G1, -psi = [|x|] on G2


@pytest.fixture(scope="module")
def hs():
    src = os.path.join(ROOT, "tests", "hostsim", "hostsim_fold_pre.cpp")
    so = os.path.join(ROOT, "tests", "hostsim", "_hostsim_fold_pre.so")
    csrc = os.path.join(ROOT, "ripp_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-shared", "-fPIC", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _fold(hs, group, p, lo, k):
    enc, dec, w = (C.g1_enc, C.g1_dec, 24) if group == 1 else (C.g2_enc, C.g2_dec, 48)
    pw, lw = np.ascontiguousarray(enc(p), np.uint32), np.ascontiguousarray(enc(lo), np.uint32)
    kw = np.ascontiguousarray(C.scalar_words(k), np.uint32)
    out = np.zeros(w, np.uint32)
    hs.hs_pre_fold(group, _ptr(pw), _ptr(lw), _ptr(kw), _ptr(out))
    return dec(out)


def _split(hs, group, k):
    kw = np.ascontiguousarray(C.scalar_words(k), np.uint32)
    out = np.zeros(56, np.uint32)
    hs.hs_endo_split(group, _ptr(kw), _ptr(out))
    pos, neg, nbits = out[:24].reshape(8, 3), out[24:48].reshape(8, 3), [int(v) for v in out[48:]]
    val = lambda words: sum(int(x) << (32 * i) for i, x in enumerate(words))
    return [val(pos[t]) - val(neg[t]) for t in range(8)], [val(pos[t]) & val(neg[t]) for t in range(8)], nbits


def _groups():
    p1, l1 = E.g1_mul(E.G1_GEN, 17), E.g1_mul(E.G1_GEN, 19)
    p2, l2 = E.g2_mul(E.G2_GEN, 17), E.g2_mul(E.G2_GEN, 19)
    return {1: (p1, l1, E.g1_mul, E.g1_add, E.g1_neg), 2: (p2, l2, E.g2_mul, E.g2_add, E.g2_neg)}


# full-width random scalars; the scalars test_xt_lane_team_folds uses to leave parts empty; scalars whose NAF carries
# across bit H (a digit of all ones below H, digits just under the base, whose NAF has one position more than bits);
# 0, 1, r - 1
CARRY = [
    (1 << 64) - 1, ((1 << 64) - 1) * LAM + (1 << 64) - 1, LAM - 1, (LAM - 1) * LAM + LAM - 1, (1 << 63) + (1 << 62),
    (1 << 32) - 1, sum(((1 << 32) - 1) * E.X_ABS**i for i in range(4)), E.X_ABS - 1, (E.X_ABS**3 - 1) + 5 * E.X_ABS**3,
    (3 << 30) * (1 + E.X_ABS + E.X_ABS**2),
]
SCALARS = [rnd.randrange(E.R) for _ in range(4)] + [E.X_ABS, E.X_ABS**2 - 1, E.X_ABS**3 + 5, 2] + CARRY + [0, 1, E.R - 1]


@pytest.mark.parametrize("group", [1, 2])
def test_split_recoding_is_exact(hs, group):
    """Part 2j + s holds NAF digits of endomorphism digit j below (s = 0) or from (s = 1) bit H: the parts recombine to
    k mod r, no digit is both +1 and -1, and every part fits the H + 1 digits the fold walks."""
    carried = False
    for k in SCALARS:
        vals, clash, nbits = _split(hs, group, k)
        parts = 4 if group == 1 else 8
        assert all(v == 0 for v in vals[parts:]) and not any(clash)
        assert all(0 <= nb <= H[group] + 1 for nb in nbits)
        assert all(nbits[t] <= H[group] for t in range(0, parts, 2)), nbits
        total = sum(vals[t] * (1 << (H[group] * (t & 1))) * BASE[group] ** (t >> 1) for t in range(parts))
        assert total % E.R == k % E.R, k
        carried |= any(nbits[t] == H[group] + 1 for t in range(1, parts, 2))
    assert carried  # some scalar's high part starts with the carry of its NAF


@pytest.mark.parametrize("group", [1, 2])
def test_pre_fold_matches_oracle(hs, group):
    p, lo, mul, add, neg = _groups()[group]
    for k in SCALARS:
        assert _fold(hs, group, p, lo, k) == add(mul(p, k), lo), k


@pytest.mark.parametrize("group", [1, 2])
def test_pre_fold_exceptional(hs, group):
    """hi or lo the identity; lo = -k hi (the sum is the identity) and lo = k hi (a doubling inside the combine)."""
    p, lo, mul, add, neg = _groups()[group]
    for k in (rnd.randrange(E.R), (1 << 64) - 1, 12345):
        assert _fold(hs, group, None, lo, k) == lo
        assert _fold(hs, group, p, None, k) == mul(p, k)
        assert _fold(hs, group, p, neg(mul(p, k)), k) is None
        assert _fold(hs, group, p, mul(p, k), k) == mul(p, 2 * k)
    assert _fold(hs, group, None, None, rnd.randrange(E.R)) is None
