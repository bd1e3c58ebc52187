"""ripp_b200/csrc/serde.cuh -- the point decoders of the deserialisation kernels -- compiled for the host (emulated carry
flag, as tests/test_hostsim.py does for the arithmetic headers) against the Python oracle's de_g1 / de_g2."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import serde as S
from oracle import serde_cases as SC
from ripp_b200 import codec as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hs():
    src = os.path.join(ROOT, "tests", "hostsim", "hostsim_serde.cpp")
    so = os.path.join(ROOT, "tests", "hostsim", "_hostsim_serde.so")
    csrc = os.path.join(ROOT, "ripp_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def _decode(hs, group, data, compressed):
    buf = np.frombuffer(data, dtype=np.uint8).copy()
    out = np.zeros(24 if group == 1 else 48, dtype=np.uint32)
    fn = hs.hs_g1_decode if group == 1 else hs.hs_g2_decode
    st = fn(ctypes.c_void_p(buf.ctypes.data), int(compressed), ctypes.c_void_p(out.ctypes.data))
    return out, st


@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("compressed", [True, False])
def test_decoder_matches_oracle(hs, group, compressed):
    de = S.de_g1 if group == 1 else S.de_g2
    enc = C.g1_enc if group == 1 else C.g2_enc
    batch = SC.mixed_batch(group, compressed, 96)
    seen = set()
    for i, b in enumerate(batch):
        want_pt, want_st = de(b, compressed)
        got, st = _decode(hs, group, b, compressed)
        assert st == want_st, (i, S.STATUS_NAMES[st], S.STATUS_NAMES[want_st])
        assert np.array_equal(got, enc(want_pt)), i
        seen.add(st)
    assert seen == set(range(5))


def test_fq2_order_and_sqrt(hs):
    half = (E.P - 1) // 2
    cases = [(0, 0), (1, 0), (half, 0), (half + 1, 0), (E.P - 1, 0), (0, 1), (0, half), (0, half + 1), (5, E.P - 1),
             (E.P - 1, 1), (half + 1, half)]
    for y in cases:
        want = (y[1] > half) if y[1] else (y[0] > half)
        assert bool(hs.hs_fq2_lex_largest(ctypes.c_void_p(np.ascontiguousarray(C.fq2_enc(y)).ctypes.data))) == want, y
    # square roots of squares with c1 = 0 (c0 a square and a non-square of Fq) and of general squares
    for a in [(4, 0), (E.P - 4, 0), (0, 0), (7, 0), (3, 9), E.f2_sqr((12345, 678))]:
        r = np.zeros(24, dtype=np.uint32)
        av = np.ascontiguousarray(C.fq2_enc(a))
        ok = hs.hs_fq2_sqrt(ctypes.c_void_p(av.ctypes.data), ctypes.c_void_p(r.ctypes.data))
        root = C.fq2_dec(r)
        if ok:
            assert E.f2_sqr(root) == (a[0] % E.P, a[1] % E.P), a
        else:
            from oracle.synth import _fp2_sqrt

            assert _fp2_sqrt(a) is None, a
