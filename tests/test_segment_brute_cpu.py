"""CPU tests for pc_segment_nearest_batch: the NULL-handle refusal, and the segment checker (tests/segment_brute.c) against a
numpy restatement of the contract's expression."""
import numpy as np

from pointcloudtraj_b200 import _lib as L
from segment_brute import brute_segment, numpy_segment_d2


def test_segment_null_handle_is_rejected():
    lib = L.load()
    assert lib.pc_segment_nearest_batch(None, None, None, 0, 3, L.PC_HOST, 0, -1.0, None, None) == L.PC_EINVAL


def _check(pts, a, b, r=None):
    gi, gd = brute_segment(pts, a, b, r)
    for j in range(len(a)):
        s = numpy_segment_d2(pts, a[j], b[j])
        ids = np.arange(len(pts))
        if r is not None:
            keep = s <= r * r
            s, ids = s[keep], ids[keep]
        if len(s) == 0:
            assert gi[j] == -1 and np.isinf(gd[j]), (j, gi[j], gd[j])
            continue
        o = np.lexsort((ids, s))[0]
        assert gi[j] == ids[o] and gd[j] == s[o], (j, gi[j], gd[j], ids[o], s[o])


def test_brute_segment_random_equals_numpy():
    rng = np.random.default_rng(4)
    pts = rng.uniform(-5, 5, (3000, 3)).astype(np.float32)
    a = rng.uniform(-6, 6, (60, 3)).astype(np.float32)
    b = (a + rng.normal(0, 3, (60, 3))).astype(np.float32)
    b[:5] = a[:5]                                       # degenerate segments
    for r in (None, 0.4, 2.0):
        _check(pts, a, b, r)


def test_brute_segment_lattice_equals_numpy():
    # segments along lattice lines and through lattice points: many d2 = 0 and exact ties, the lowest index wins
    g = np.arange(8, dtype=np.float32) * 0.5
    pts = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    pts = np.concatenate([pts, pts[::-1]]).astype(np.float32)      # every point twice
    a = np.array([[0, 0, 0], [0, 1, 1], [0.25, 0.25, 0.25], [-1, -1, -1], [3.5, 0, 0], [1, 1, 1]], np.float32)
    b = np.array([[3.5, 0, 0], [3.5, 1, 1], [3.25, 3.25, 3.25], [-1, -1, 5], [3.5, 0, 0], [2, 2.5, 0.5]], np.float32)
    for r in (None, 0.25, 1.0):
        _check(pts, a, b, r)
    gi, gd = brute_segment(pts, a[:2], b[:2])
    assert (gd == 0).all() and gi[0] == 0, (gi, gd)


def test_brute_segment_nonfinite_and_empty():
    pts = np.zeros((4, 3), np.float32)
    a = np.array([[np.nan, 0, 0], [0, 0, 0], [0, np.inf, 0]], np.float32)
    b = np.array([[1, 0, 0], [1, 0, 0], [0, 0, 0]], np.float32)
    gi, gd = brute_segment(pts, a, b)
    assert gi.tolist() == [-1, 0, -1] and np.isnan(gd[[0, 2]]).all() and gd[1] == 0
    gi, gd = brute_segment(pts[:0], a[1:2], b[1:2])
    assert gi[0] == -1 and np.isinf(gd[0])
