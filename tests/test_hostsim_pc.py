"""The Fr rules of the polynomial-commitment kernels (ripp_b200/csrc/pc_scan.cuh: the chunked division scan of
k_pc_div_heads / k_pc_div_replay, its carry combine, and the Horner step of k_pc_rows / k_pc_rows_combine) compiled for
the host and compared with the oracle's synthetic division and evaluation (oracle/poly_commit.py)."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import poly_commit as OPC
from ripp_b200 import codec as C
from ripp_b200.poly_commit import quotient_by_linear

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hs():
    src = os.path.join(ROOT, "tests", "hostsim", "hostsim_pc.cpp")
    so = os.path.join(ROOT, "tests", "hostsim", "_hostsim_pc.so")
    csrc = os.path.join(ROOT, "ripp_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".h"))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _div(hs, coeffs, z, L):
    c = C.fr_vec_enc(coeffs) if coeffs else np.zeros((1, 8), dtype=np.uint32)
    q = np.zeros((max(len(coeffs) - 1, 1), 8), dtype=np.uint32)
    ev, zw = np.zeros(8, dtype=np.uint32), C.fr_enc(z)
    hs.hs_div_linear(_ptr(c), ctypes.c_size_t(len(coeffs)), _ptr(zw), ctypes.c_size_t(L), _ptr(q), _ptr(ev))
    return [C.fr_dec(w) for w in q[: max(len(coeffs) - 1, 0)]], C.fr_dec(ev)


def _lengths(L):
    out = {0, 1, 2, L - 1, L, L + 1, L * L - 1, L * L, L * L + 1, L * L * L + 1}
    for k in (5, 8, 11):
        out |= {(1 << k) - 1, 1 << k, (1 << k) + 1}
    return sorted(n for n in out if n >= 0)


@pytest.mark.parametrize("L", [2, 3, 8, 32])
def test_division_scan_matches_oracle(hs, L):
    rnd = random.Random(L)
    for n in _lengths(L):
        coeffs = [rnd.randrange(E.R) for _ in range(n)]
        for z in (0, 1, E.R - 1, rnd.randrange(E.R)):
            q, ev = _div(hs, coeffs, z, L)
            assert q == quotient_by_linear(coeffs, z) == OPC.quotient_by_linear(coeffs, z), (L, n, z)
            assert ev == OPC.poly_eval(coeffs, z), (L, n, z)


def test_carry_combine_is_the_recurrence_at_z_pow_l(hs):
    """S_b = head_b + z^L S_(b+1): the value at a chunk's start from its head and the next chunk's start."""
    rnd = random.Random(5)
    L, z = 4, rnd.randrange(E.R)
    coeffs = [rnd.randrange(E.R) for _ in range(3 * L)]
    s = [OPC.poly_eval(coeffs[k:], z) for k in range(len(coeffs))]  # s_k = sum_(i >= k) c_i z^(i - k)
    for b in range(2):
        head = OPC.poly_eval(coeffs[b * L:(b + 1) * L], z)
        out, args = np.zeros(8, dtype=np.uint32), [C.fr_enc(head), C.fr_enc(pow(z, L, E.R)), C.fr_enc(s[(b + 1) * L])]
        hs.hs_carry_combine(*[_ptr(a) for a in args], _ptr(out))
        assert C.fr_dec(out) == s[b * L]


@pytest.mark.parametrize("n,m,R,len_", [(8, 8, 1, 64), (8, 8, 3, 61), (16, 4, 5, 37), (4, 16, 4, 0), (1, 8, 1, 5), (64, 2, 7, 128)])
def test_row_combination_matches_oracle(hs, n, m, R, len_):
    rnd = random.Random(n * 1000 + m * 10 + R)
    flat = [rnd.randrange(E.R) for _ in range(len_)]
    x = rnd.randrange(E.R)
    words = C.fr_vec_enc(flat) if flat else np.zeros((1, 8), dtype=np.uint32)
    y, xw = np.zeros((m, 8), dtype=np.uint32), C.fr_enc(x)
    hs.hs_rows(_ptr(words), ctypes.c_size_t(len_), ctypes.c_size_t(m), ctypes.c_size_t(n), ctypes.c_size_t(R), _ptr(xw), _ptr(y))
    padded = flat + [0] * (n * m - len_)
    want = [sum(pow(x, i, E.R) * padded[i * m + j] for i in range(n)) % E.R for j in range(m)]
    assert [C.fr_dec(w) for w in y] == want
    # and y_eval(y) is the bivariate evaluation (mod.rs:137-150)
    yy = rnd.randrange(E.R)
    rows = [padded[i * m:(i + 1) * m] for i in range(n)]
    assert OPC.poly_eval(want, yy) == OPC.bivariate_evaluate(rows, (x, yy))
