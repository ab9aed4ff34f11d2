"""CPU tests for pc_knn_large_batch: the NULL-handle refusal, and the kNN checker (tests/knn_brute.c) at the row lengths of
the large call."""
import numpy as np

from knn_brute import brute_knn
from pointcloudtraj_b200 import _lib as L


def test_knn_large_null_handle_is_rejected():
    lib = L.load()
    assert lib.pc_knn_large_batch(None, None, 0, 3, L.PC_HOST, 0, 64, -1.0, None, None) == L.PC_EINVAL


def test_brute_knn_k1024_equals_lexsort():
    rng = np.random.default_rng(3)
    # a coarse lattice: many equal distances, duplicated points, and fewer points than k for the padding
    pts = (rng.integers(0, 9, size=(1500, 3)) * 0.25).astype(np.float32)
    q = np.concatenate([pts[:10], rng.uniform(-0.5, 2.5, (20, 3))]).astype(np.float32)
    P = pts.astype(np.float64)
    for n, k, r in ((1500, 1024, None), (1500, 1024, 0.6), (700, 1024, None), (1500, 33, None)):
        gi, gd = brute_knn(pts[:n], q, k, r)
        for j in range(len(q)):
            d = P[:n] - q[j].astype(np.float64)
            s = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
            ids = np.arange(n)
            if r is not None:
                keep = s <= r * r
                s, ids = s[keep], ids[keep]
            o = np.lexsort((ids, s))[:k]
            assert gi[j, : len(o)].tolist() == ids[o].tolist() and (gd[j, : len(o)] == s[o]).all(), (n, k, r, j)
            assert (gi[j, len(o):] == -1).all() and np.isinf(gd[j, len(o):]).all()
