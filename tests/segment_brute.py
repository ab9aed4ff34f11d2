"""TEST INFRASTRUCTURE ONLY: fp64 brute-force nearest point to a segment (segment_brute.c), the arbiter of the segment tests.

The C file is compiled on first use into a temporary directory (the repository tree is never written), with the flags of
knn_brute.py: -O2 -ffp-contract=off (un-fused fp64 in the contract's operation order) -fopenmp (segments in parallel).
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
        d = tempfile.mkdtemp(prefix="pc_segment_brute_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsegment_brute.so")
        out = subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-std=gnu11", "-o", so,
                              os.path.join(_HERE, "segment_brute.c"), "-lm"], capture_output=True, text=True)
        if out.returncode != 0:
            raise RuntimeError("compiling tests/segment_brute.c failed:\n" + out.stdout + out.stderr)
        L = C.CDLL(so)
        f32p, i64p, f64p = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_double)
        L.segment_brute_batch.argtypes = [f32p, C.c_int64, C.c_int64, f32p, f32p, C.c_int64, C.c_int64, C.c_double, i64p, f64p, C.c_int]
        L.segment_d2.argtypes = [f32p, f32p, f32p]
        L.segment_d2.restype = C.c_double
        _lib = L
    return _lib


def _rows(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4):
        raise ValueError("expected an (n, 3) or (n, 4) float32 array")
    return a


def brute_segment(xyz, a, b, max_range=None, nthreads=0):
    """The smallest (fp64 d2, original index) per segment [a[j], b[j]]; with max_range only points with d2 <= max_range**2.
    Returns (idx int64[m], d2 float64[m]): -1 / inf without a point, -1 / NaN for a non-finite endpoint."""
    xyz, a, b = _rows(xyz), _rows(a), _rows(b)
    if a.shape != b.shape:
        raise ValueError("a and b need the same shape")
    m = a.shape[0]
    idx = np.empty(m, dtype=np.int64)
    d2 = np.empty(m, dtype=np.float64)
    r = -1.0 if max_range is None else float(max_range)
    f32p, i64p, f64p = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_double)
    _load().segment_brute_batch(xyz.ctypes.data_as(f32p), xyz.shape[0], xyz.shape[1], a.ctypes.data_as(f32p), b.ctypes.data_as(f32p),
                                m, a.shape[1], r, idx.ctypes.data_as(i64p), d2.ctypes.data_as(f64p), int(nthreads))
    return idx, d2


def numpy_segment_d2(P, a, b):
    """The contract's expression restated in numpy float64 (elementwise IEEE operations, no fusion): d2 of every point of P
    (n, 3) to one segment [a, b]."""
    P = np.asarray(P, np.float32)[:, :3].astype(np.float64)
    A = np.asarray(a, np.float32)[:3].astype(np.float64)
    B = np.asarray(b, np.float32)[:3].astype(np.float64)
    D = B - A
    W = P - A
    L2 = (D[0] * D[0] + D[1] * D[1]) + D[2] * D[2]
    s = (W[:, 0] * D[0] + W[:, 1] * D[1]) + W[:, 2] * D[2]
    WB = P - B
    dA = (W[:, 0] * W[:, 0] + W[:, 1] * W[:, 1]) + W[:, 2] * W[:, 2]
    dB = (WB[:, 0] * WB[:, 0] + WB[:, 1] * WB[:, 1]) + WB[:, 2] * WB[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        t = s / L2
    E = W - t[:, None] * D[None, :]
    dE = (E[:, 0] * E[:, 0] + E[:, 1] * E[:, 1]) + E[:, 2] * E[:, 2]
    return np.where((s <= 0.0) | (L2 == 0.0), dA, np.where(s >= L2, dB, dE))
