"""ORACLE side: build + ctypes binding of the compiled CPU restatement of validated point decoding
(oracle/cpu/serde_cpu.cpp, the rules of oracle/serde.py), OpenMP over the elements."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "serde_cpu.cpp")
OUT_DIR = os.path.join(HERE, "_build")
LIB = os.path.join(OUT_DIR, "libripp_cpu_serde.so")

_lib = None


def build(force=False):
    deps = [SRC] + [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith(".hpp")]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in deps):
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    # -march=x86-64-v3 (not native): the .so built here must run on the GPU box's host CPU
    cmd = ["g++", "-O3", "-std=c++17", "-march=x86-64-v3", "-fopenmp", "-shared", "-fPIC", "-o", LIB, SRC]
    subprocess.run(cmd, check=True)
    return LIB


def load():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(LIB)
        _lib.cpu_serde_threads.restype = ctypes.c_int
    return _lib


def threads():
    return load().cpu_serde_threads()


def deserialize(group, data, n, stride, compressed):
    """Validated decoding of n ark-serialize points (group 1 / 2) at `stride` bytes.  -> (points (n, 24 | 48) uint32
    Montgomery words as include/ripp_b200.h lays them out, all zero for the identity and rejected elements; status (n,)
    uint8 in oracle/serde.py's numbering)."""
    lib = load()
    buf = np.frombuffer(bytes(data), dtype=np.uint8).copy() if len(data) else np.zeros(1, dtype=np.uint8)
    pts = np.zeros((n, 24 if group == 1 else 48), dtype=np.uint32)
    st = np.zeros(n, dtype=np.uint8)
    fn = lib.cpu_g1_deserialize if group == 1 else lib.cpu_g2_deserialize
    p = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731
    fn(p(buf), ctypes.c_size_t(n), ctypes.c_size_t(stride), int(bool(compressed)), p(pts), p(st))
    return pts, st
