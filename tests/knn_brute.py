"""TEST INFRASTRUCTURE ONLY: fp64 brute-force k nearest neighbours (knn_brute.c), the arbiter of the kNN tests.

The C file is compiled on first use into a temporary directory (the repository tree is never written), with the flags of
the oracle's build: -O2 -ffp-contract=off (un-fused fp64 in the reference's operation order) -fopenmp (queries in parallel).
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _load():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="pc_knn_brute_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libknn_brute.so")
        out = subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-std=gnu11", "-o", so,
                              os.path.join(_HERE, "knn_brute.c"), "-lm"], capture_output=True, text=True)
        if out.returncode != 0:
            raise RuntimeError("compiling tests/knn_brute.c failed:\n" + out.stdout + out.stderr)
        L = C.CDLL(so)
        f32p, i64p, f64p = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_double)
        L.knn_brute_batch.argtypes = [f32p, C.c_int64, C.c_int64, f32p, C.c_int64, C.c_int64, C.c_int, C.c_double, i64p, f64p, C.c_int]
        _lib = L
    return _lib


def _rows(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4):
        raise ValueError("expected an (n, 3) or (n, 4) float32 array")
    return a


def brute_knn(xyz, q, k, max_range=None, nthreads=0):
    """The k smallest (fp64 d2, original index) per query in the reference's operation order; with max_range only points
    with d2 <= max_range**2.  Returns (idx int64[m, k], d2 float64[m, k]), rows padded with -1 / inf."""
    xyz, q, k = _rows(xyz), _rows(q), int(k)
    if k < 1:
        raise ValueError("k must be >= 1")
    m = q.shape[0]
    idx = np.empty((m, k), dtype=np.int64)
    d2 = np.empty((m, k), dtype=np.float64)
    r = -1.0 if max_range is None else float(max_range)
    f32p, i64p, f64p = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_double)
    _load().knn_brute_batch(xyz.ctypes.data_as(f32p), xyz.shape[0], xyz.shape[1], q.ctypes.data_as(f32p), m, q.shape[1], k, r,
                            idx.ctypes.data_as(i64p), d2.ctypes.data_as(f64p), int(nthreads))
    return idx, d2
