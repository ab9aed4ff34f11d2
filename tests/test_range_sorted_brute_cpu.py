"""CPU tests of the sorted-range checker (tests/range_sorted_brute.c) and of pc_range_sorted_batch's argument
checks that need no GPU."""
import numpy as np

import oracle
from knn_brute import brute_knn
from range_sorted_brute import brute_range_sorted
from pointcloudtraj_b200 import _lib as L
from pointcloudtraj_b200 import synth


def _lexsort_rows(pts, q, r, max_nn):
    """numpy restatement: every point with oracle.pair_d2 <= r**2, np.lexsort by (d2, index), cut to max_nn."""
    rr = np.broadcast_to(np.atleast_1d(np.asarray(r, np.float64)), (len(q),))
    ids_all = np.arange(len(pts))
    rows = []
    for j in range(len(q)):
        s = oracle.pair_d2(pts, np.repeat(q[j:j + 1], len(pts), 0), ids_all)
        ids = ids_all[s <= rr[j] * rr[j]]
        s = s[s <= rr[j] * rr[j]]
        o = np.lexsort((ids, s))
        if max_nn:
            o = o[:max_nn]
        rows.append((ids[o], s[o]))
    return rows


def _tie_heavy(n, seed):
    rng = np.random.default_rng(seed)
    pts = (rng.integers(0, 5, size=(n, 3)) * 0.25).astype(np.float32)
    q = np.concatenate([(rng.integers(0, 5, size=(30, 3)) * 0.25), (rng.integers(0, 9, size=(30, 3)) * 0.125)]).astype(np.float32)
    return pts, q


def test_brute_range_sorted_equals_lexsort():
    for seed in range(2):
        pts, q = _tie_heavy(400, seed)
        per_query = np.random.default_rng(seed).uniform(0.0, 0.6, len(q))
        for r in (0.3, 0.0, per_query):
            for max_nn in (0, 1, 7, 40):
                off, idx, d2 = brute_range_sorted(pts, q, r, max_nn)
                for j, (ei, ed) in enumerate(_lexsort_rows(pts, q, r, max_nn)):
                    gi, gd = idx[off[j]:off[j + 1]], d2[off[j]:off[j + 1]]
                    assert gi.tolist() == ei.tolist() and (gd == ed).all(), (seed, max_nn, j)


def test_brute_range_sorted_equals_brute_knn():
    pts, half = synth.forest_cloud(20000, seed=4, variant="L", return_half=True)
    q = synth.rrt_queries(300, half, seed=5, lattice_frac=0.5)
    r = 0.45
    for k in (1, 8, 32):
        off, idx, d2 = brute_range_sorted(pts, q, r, k)
        ki, kd = brute_knn(pts, q, k, r)
        for j in range(len(q)):
            n = off[j + 1] - off[j]
            assert (ki[j, :n] == idx[off[j]:off[j + 1]]).all() and (kd[j, :n] == d2[off[j]:off[j + 1]]).all()
            assert (ki[j, n:] == -1).all()


def test_brute_range_sorted_degenerate():
    pts = np.zeros((5, 3), np.float32)
    off, idx, d2 = brute_range_sorted(pts, np.zeros((2, 3), np.float32), [float("nan"), 0.0])
    assert off.tolist() == [0, 0, 5] and idx.tolist() == [0, 1, 2, 3, 4] and (d2 == 0).all()
    off, idx, d2 = brute_range_sorted(np.zeros((0, 3), np.float32), np.zeros((3, 3), np.float32), 1.0)
    assert off.tolist() == [0, 0, 0, 0] and len(idx) == 0
    off, idx, d2 = brute_range_sorted(pts, np.zeros((0, 3), np.float32), 1.0)
    assert off.tolist() == [0] and len(idx) == 0


def test_range_sorted_null_handle_is_rejected():
    lib = L.load()
    assert lib.pc_range_sorted_batch(None, None, 0, 3, L.PC_HOST, None, 1, 0, None, None, None, 0) == L.PC_EINVAL
