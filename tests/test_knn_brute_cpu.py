"""CPU tests of the kNN checker (tests/knn_brute.c) and of pc_knn_batch's argument checks that need no GPU."""
import numpy as np

import oracle
from knn_brute import brute_knn
from pointcloudtraj_b200 import _lib as L
from pointcloudtraj_b200 import synth


def _lexsort_knn(pts, q, k, max_range=None):
    """numpy restatement: fp64 d2 in the reference's order, np.lexsort by (d2, index), cut to k, padded."""
    P = pts.astype(np.float64)
    idx = np.full((len(q), k), -1, np.int64)
    d2 = np.full((len(q), k), np.inf)
    for j in range(len(q)):
        d = P - q[j].astype(np.float64)
        s = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        ids = np.arange(len(P))
        if max_range is not None:
            keep = s <= max_range * max_range
            s, ids = s[keep], ids[keep]
        o = np.lexsort((ids, s))[:k]
        idx[j, : len(o)] = ids[o]
        d2[j, : len(o)] = s[o]
    return idx, d2


def _tie_heavy(n, seed):
    """Points on a coarse lattice with many duplicates, queries on lattice points and half-way between them."""
    rng = np.random.default_rng(seed)
    pts = (rng.integers(0, 5, size=(n, 3)) * 0.25).astype(np.float32)
    q = np.concatenate([(rng.integers(0, 5, size=(40, 3)) * 0.25), (rng.integers(0, 9, size=(40, 3)) * 0.125)]).astype(np.float32)
    return pts, q


def test_brute_knn_k1_equals_brute_nearest():
    pts, half = synth.forest_cloud(5000, seed=3, variant="L", return_half=True)
    q = synth.rrt_queries(500, half, seed=2, lattice_frac=0.5)
    i1, d1 = brute_knn(pts, q, 1)
    i0, d0, _ = oracle.brute_nearest(pts, q)
    assert (i1[:, 0] == i0).all() and (d1[:, 0] == d0).all()


def test_brute_knn_equals_lexsort_on_ties():
    for seed in range(3):
        pts, q = _tie_heavy(300, seed)
        for k in (1, 2, 5, 16, 32):
            for r in (None, 0.3, 0.0):
                gi, gd = brute_knn(pts, q, k, r)
                ei, ed = _lexsort_knn(pts, q, k, r)
                assert (gi == ei).all() and (gd == ed).all(), (seed, k, r)


def test_brute_knn_pads_small_clouds():
    pts = np.array([[0, 0, 0], [1, 0, 0], [0, 0, 0]], np.float32)
    idx, d2 = brute_knn(pts, np.zeros((1, 3), np.float32), 5)
    assert idx.tolist() == [[0, 2, 1, -1, -1]]
    assert d2[0, :3].tolist() == [0.0, 0.0, 1.0] and np.isinf(d2[0, 3:]).all()
    idx, d2 = brute_knn(np.zeros((0, 3), np.float32), np.zeros((2, 3), np.float32), 3)
    assert (idx == -1).all() and np.isinf(d2).all()


def test_brute_knn_bounded_equals_range_lists():
    """A bounded row is the range list re-sorted by (d2, index) and cut to k."""
    pts, half = synth.forest_cloud(20000, seed=4, variant="L", return_half=True)
    q = synth.rrt_queries(300, half, seed=5, lattice_frac=0.5)
    r = 0.45
    ko = oracle.KdOracle().build(pts, np.random.default_rng(0).permutation(len(pts)))
    off, lst = ko.range(q, r)
    for k in (4, 32):
        idx, d2 = brute_knn(pts, q, k, r)
        for j in range(len(q)):
            ids = lst[off[j]:off[j + 1]]
            s = oracle.pair_d2(pts, np.repeat(q[j:j + 1], len(ids), 0), ids)
            o = np.lexsort((ids, s))[:k]
            assert idx[j, : len(o)].tolist() == ids[o].tolist() and (d2[j, : len(o)] == s[o]).all()
            assert (idx[j, len(o):] == -1).all() and np.isinf(d2[j, len(o):]).all()


def test_knn_null_handle_is_rejected():
    lib = L.load()
    assert lib.pc_knn_batch(None, None, 0, 3, L.PC_HOST, 0, 4, -1.0, None, None) == L.PC_EINVAL
