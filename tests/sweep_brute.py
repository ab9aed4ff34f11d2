"""TEST INFRASTRUCTURE ONLY: fp64 brute-force first contact of a swept sphere (sweep_brute.c), the arbiter of the sweep tests.

The C file is compiled on first use into a temporary directory (the repository tree is never written), with the flags of
segment_brute.py: -O2 -ffp-contract=off (un-fused fp64 in the contract's operation order) -fopenmp (segments in parallel).
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
        d = tempfile.mkdtemp(prefix="pc_sweep_brute_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libsweep_brute.so")
        out = subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-std=gnu11", "-o", so,
                              os.path.join(_HERE, "sweep_brute.c"), "-lm"], capture_output=True, text=True)
        if out.returncode != 0:
            raise RuntimeError("compiling tests/sweep_brute.c failed:\n" + out.stdout + out.stderr)
        L = C.CDLL(so)
        f32p, i64p, f64p = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_double)
        L.sweep_brute_batch.argtypes = [f32p, C.c_int64, C.c_int64, f32p, f32p, C.c_int64, C.c_int64, C.c_double, i64p, f64p, C.c_int]
        _lib = L
    return _lib


def _rows(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4):
        raise ValueError("expected an (n, 3) or (n, 4) float32 array")
    return a


def brute_sweep(xyz, a, b, radius, nthreads=0):
    """The smallest (fp64 t, original index) per segment [a[j], b[j]] for a sphere of the given radius.
    Returns (idx int64[m], t float64[m]): -1 / inf without contact, -1 / NaN for a non-finite endpoint."""
    xyz, a, b = _rows(xyz), _rows(a), _rows(b)
    if a.shape != b.shape:
        raise ValueError("a and b need the same shape")
    m = a.shape[0]
    idx = np.empty(m, dtype=np.int64)
    t = np.empty(m, dtype=np.float64)
    f32p, i64p, f64p = C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_double)
    _load().sweep_brute_batch(xyz.ctypes.data_as(f32p), xyz.shape[0], xyz.shape[1], a.ctypes.data_as(f32p), b.ctypes.data_as(f32p),
                              m, a.shape[1], float(radius), idx.ctypes.data_as(i64p), t.ctypes.data_as(f64p), int(nthreads))
    return idx, t


def round_down_f32(t):
    """float64 -> float32 rounded toward -inf (what out_t holds); np.float32 rounds to nearest.  NaN and inf pass through."""
    t = np.asarray(t, np.float64)
    f = t.astype(np.float32)
    up = np.isfinite(t) & (f.astype(np.float64) > t)
    f[up] = np.nextafter(f[up], np.float32(-np.inf))
    return f


def numpy_sweep_t(P, a, b, radius):
    """The contract's expression restated in numpy float64 (elementwise IEEE operations, no fusion): t of every point of P
    (n, 3) for one segment [a, b]; +inf where a point makes no contact."""
    P = np.asarray(P, np.float32)[:, :3].astype(np.float64)
    A = np.asarray(a, np.float32)[:3].astype(np.float64)
    B = np.asarray(b, np.float32)[:3].astype(np.float64)
    r2 = np.float64(radius) * np.float64(radius)
    D = B - A
    W = P - A
    WB = P - B
    c0 = (W[:, 0] * W[:, 0] + W[:, 1] * W[:, 1]) + W[:, 2] * W[:, 2]
    cB = (WB[:, 0] * WB[:, 0] + WB[:, 1] * WB[:, 1]) + WB[:, 2] * WB[:, 2]
    L2 = (D[0] * D[0] + D[1] * D[1]) + D[2] * D[2]
    s = (W[:, 0] * D[0] + W[:, 1] * D[1]) + W[:, 2] * D[2]
    h = c0 - r2
    disc = s * s - L2 * h
    with np.errstate(divide="ignore", invalid="ignore"):
        tq = h / (s + np.sqrt(disc))
    quad = (L2 != 0.0) & (s > 0.0) & (disc >= 0.0) & (tq <= 1.0)
    return np.where(c0 <= r2, 0.0, np.where(quad, tq, np.where(cB <= r2, 1.0, np.inf)))


def numpy_quadratic_t(p, a, b, radius):
    """The quadratic branch's t' = h / (s + sqrt(disc)) of one point (NaN where disc < 0), without the branch conditions."""
    P, A, B = (np.asarray(v, np.float32)[:3].astype(np.float64) for v in (p, a, b))
    D, W = B - A, P - A
    c0 = (W[0] * W[0] + W[1] * W[1]) + W[2] * W[2]
    L2 = (D[0] * D[0] + D[1] * D[1]) + D[2] * D[2]
    s = (W[0] * D[0] + W[1] * D[1]) + W[2] * D[2]
    h = c0 - np.float64(radius) * np.float64(radius)
    disc = s * s - L2 * h
    with np.errstate(invalid="ignore"):
        return h / (s + np.sqrt(disc))


def b_clause_rows(rng, n, radius=0.3125):
    """n axis-aligned segments with one point each at exactly `radius` from b, just beyond it: (3/5, 4/5) radius along and
    across the axis, so |P - B|^2 = R2 exactly (radius = 5 * 2^-k) and the exact first contact is t = 1.  The rounded
    quadratic lands above 1 for about half of them; those reach the contact only through the B clause.
    Returns (a, b, p), float32 (n, 3) each."""
    q = np.float32(radius / 5)
    b = rng.uniform(-15, 15, (n, 3)).astype(np.float32)
    ax = rng.integers(0, 3, n)
    lat = (ax + rng.integers(1, 3, n)) % 3
    sg = rng.choice([-1.0, 1.0], n).astype(np.float32)
    a = b.copy()
    a[np.arange(n), ax] -= (sg * rng.uniform(0.5, 20, n)).astype(np.float32)
    p = b.copy()
    p[np.arange(n), ax] += sg * 3 * q
    p[np.arange(n), lat] += rng.choice([-1.0, 1.0], n).astype(np.float32) * 4 * q
    return a, b, p
