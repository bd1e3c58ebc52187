"""The batched polynomial-commitment rules (ripp_b200/csrc/pc_scan.cuh: the segmented division scan of
k_pc_div_heads_seg / k_pc_div_replay_seg and the grouped row combination of k_pc_rows_seg / k_pc_rows_combine_seg)
compiled for the host and compared with the oracle over several batch sizes and chunk lengths, and the batch grouping
over the batch shapes the entry points accept, the corner of 2^16 rows of one included."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import poly_commit as OPC
from ripp_b200 import codec as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROW_THREADS = 1 << 16


@pytest.fixture(scope="module")
def hs():
    src = os.path.join(ROOT, "tests", "hostsim", "hostsim_pc_batch.cpp")
    so = os.path.join(ROOT, "tests", "hostsim", "_hostsim_pc_batch.so")
    csrc = os.path.join(ROOT, "ripp_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".h"))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _enc(vals):
    return C.fr_vec_enc(vals) if vals else np.zeros((1, 8), dtype=np.uint32)


@pytest.mark.parametrize("log_l", [1, 2, 3, 5])
@pytest.mark.parametrize("count", [1, 3, 8])
def test_segmented_division_matches_oracle(hs, log_l, count):
    L = 1 << log_l
    rnd = random.Random(100 * count + log_l)
    for N in sorted({1, 2, L - 1, L, L + 1, L * L + 3, 64, 129}):
        if N < 1:
            continue
        polys = [[rnd.randrange(E.R) for _ in range(N)] for _ in range(count)]
        zs = [[0, 1, E.R - 1][k] if k < 3 else rnd.randrange(E.R) for k in range(count)]
        c = np.ascontiguousarray(np.concatenate([_enc(p) for p in polys]))
        z = np.ascontiguousarray(_enc(zs))
        q = np.zeros((count * N, 8), dtype=np.uint32)
        ev = np.zeros((count, 8), dtype=np.uint32)
        hs.hs_div_batch(_ptr(c), ctypes.c_size_t(count), ctypes.c_size_t(N), _ptr(z), ctypes.c_uint(log_l), _ptr(q), _ptr(ev))
        for k in range(count):
            got_q = [C.fr_dec(w) for w in q[k * N:k * N + N - 1]]
            assert got_q == OPC.quotient_by_linear(polys[k], zs[k]), (L, N, k)
            assert C.fr_dec(ev[k]) == OPC.poly_eval(polys[k], zs[k]), (L, N, k)


def _groups(hs, count, n, m):
    G, R, B = ctypes.c_size_t(), ctypes.c_size_t(), ctypes.c_size_t()
    hs.hs_row_groups_batch(ctypes.c_size_t(count), ctypes.c_size_t(n), ctypes.c_size_t(m), ctypes.byref(G), ctypes.byref(R),
                           ctypes.byref(B))
    return G.value, R.value, B.value


def test_row_groups_over_batch_shapes(hs):
    """Every count, n, m with count n <= 2^16 and count n m <= 2^24 (powers of two, and count 3 and 5 in between):
    full non-empty groups, about ROW_THREADS threads, and a one-dimensional grid within CUDA's 2^31 - 1 blocks."""
    for ln in range(17):
        for lm in range(25 - ln):
            n, m = 1 << ln, 1 << lm
            for count in sorted({1, 2, 3, 5, 16, 1 << 10, (1 << 16) // n, (1 << 24) // (n * m)}):
                if count < 1 or count * n > 1 << 16 or count * n * m > 1 << 24:
                    continue
                G, R, B = _groups(hs, count, n, m)
                assert 1 <= G <= n and G * R >= n > (G - 1) * R, (count, n, m)
                assert B == (count * G * m + 127) // 128 and B <= 2 ** 31 - 1, (count, n, m)
                assert count * G * m <= max(ROW_THREADS, count * m), (count, n, m)
                if count * m < ROW_THREADS and G < n:
                    assert 2 * count * G * m > ROW_THREADS // 2, (count, n, m)  # a full GPU's worth of threads


def test_row_index_covers_every_thread_once(hs):
    for count, G, m in [(3, 4, 8), (5, 1, 1), (2, 7, 2)]:
        seen = set()
        for i in range(count * G * m):
            k, g, j = ctypes.c_size_t(), ctypes.c_size_t(), ctypes.c_size_t()
            hs.hs_row_index(ctypes.c_size_t(i), ctypes.c_size_t(G), ctypes.c_size_t(m), ctypes.byref(k), ctypes.byref(g), ctypes.byref(j))
            assert (k.value * G + g.value) * m + j.value == i
            seen.add((k.value, g.value, j.value))
        assert len(seen) == count * G * m


@pytest.mark.parametrize("count,n,m", [(1, 8, 4), (3, 8, 4), (8, 16, 1), (5, 4, 16), (3, 1, 8), (1 << 12, 16, 1), (2, 1024, 2)])
def test_batched_row_combination_matches_oracle(hs, count, n, m):
    rnd = random.Random(count * 7 + n + m)
    nm = n * m
    lens = [[0, 1, nm - m, m + 1 if nm > m + 1 else nm, nm][k % 5] for k in range(count)]
    lens = [max(0, min(nm, x)) for x in lens]
    polys = [[rnd.randrange(E.R) for _ in range(x)] for x in lens]
    offs = np.cumsum([0] + lens[:-1]).astype(np.uintp)
    flat = [v for p in polys for v in p]
    c = np.ascontiguousarray(_enc(flat))
    xs = [[0, 1, E.R - 1][k] if k < 3 else rnd.randrange(E.R) for k in range(count)]
    x = np.ascontiguousarray(_enc(xs))
    y = np.zeros((count * m, 8), dtype=np.uint32)
    ln = np.ascontiguousarray(np.array(lens, dtype=np.uintp))
    offs = np.ascontiguousarray(offs)
    hs.hs_rows_batch(_ptr(c), _ptr(offs), _ptr(ln), ctypes.c_size_t(count), ctypes.c_size_t(n), ctypes.c_size_t(m), _ptr(x), _ptr(y))
    for k in sorted({0, 1, 2, count - 1} & set(range(count))):
        full = polys[k] + [0] * (nm - lens[k])
        rows = [full[i * m:(i + 1) * m] for i in range(n)]
        want = [sum(rows[i][j] * pow(xs[k], i, E.R) for i in range(n)) % E.R for j in range(m)]
        assert [C.fr_dec(w) for w in y[k * m:(k + 1) * m]] == want, (count, n, m, k)
