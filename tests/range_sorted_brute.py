"""TEST INFRASTRUCTURE ONLY: fp64 brute-force sorted range lists (range_sorted_brute.c), the arbiter of the sorted-range tests.

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
        d = tempfile.mkdtemp(prefix="pc_range_sorted_brute_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "librange_sorted_brute.so")
        out = subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-std=gnu11", "-o", so,
                              os.path.join(_HERE, "range_sorted_brute.c"), "-lm"], capture_output=True, text=True)
        if out.returncode != 0:
            raise RuntimeError("compiling tests/range_sorted_brute.c failed:\n" + out.stdout + out.stderr)
        L = C.CDLL(so)
        f32p, i64p, f64p = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_double)
        L.range_sorted_brute.argtypes = [f32p, C.c_int64, C.c_int64, f32p, C.c_int64, C.c_int64, f64p, C.c_int, C.c_int64,
                                         i64p, i64p, i64p, f64p, C.c_int]
        _lib = L
    return _lib


def _rows(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4):
        raise ValueError("expected an (n, 3) or (n, 4) float32 array")
    return a


def brute_range_sorted(xyz, q, r, max_nn=0, nthreads=0):
    """Every point with d2 <= r**2 per query (r: one radius or one per query), in the reference's operation order, sorted by
    (fp64 d2, original index) and cut to max_nn (0 keeps all).  Returns (offsets int64[m+1], idx int64[total], d2 float64[total])."""
    xyz, q, max_nn = _rows(xyz), _rows(q), int(max_nn)
    if max_nn < 0:
        raise ValueError("max_nn must be >= 0")
    m = q.shape[0]
    rr = np.ascontiguousarray(np.atleast_1d(r), dtype=np.float64)
    scalar = 1 if rr.shape[0] == 1 else 0
    if not scalar and rr.shape[0] != m:
        raise ValueError("need one radius or one per query")
    f32p, i64p, f64p = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_double)
    lib = _load()
    args = (xyz.ctypes.data_as(f32p), xyz.shape[0], xyz.shape[1], q.ctypes.data_as(f32p), m, q.shape[1], rr.ctypes.data_as(f64p),
            scalar, max_nn)
    counts = np.zeros(max(m, 1), dtype=np.int64)
    null64, nullf = C.POINTER(C.c_int64)(), C.POINTER(C.c_double)()
    if lib.range_sorted_brute(*args, counts.ctypes.data_as(i64p), null64, null64, nullf, int(nthreads)) != 0:
        raise RuntimeError("range_sorted_brute failed")
    off = np.zeros(m + 1, dtype=np.int64)
    off[1:] = np.cumsum(counts[:m])
    idx = np.empty(max(int(off[-1]), 1), dtype=np.int64)
    d2 = np.empty(max(int(off[-1]), 1), dtype=np.float64)
    if lib.range_sorted_brute(*args, null64, off.ctypes.data_as(i64p), idx.ctypes.data_as(i64p), d2.ctypes.data_as(f64p), int(nthreads)) != 0:
        raise RuntimeError("range_sorted_brute failed")
    return off, idx[: off[-1]], d2[: off[-1]]
