"""GPU tests of pc_knn_batch: bit-equal with the fp64 brute force (tests/knn_brute.c) on both forced paths (one warp per query,
curve-ordered packets) and in both memory spaces, plus the relations to pc_nearest_batch and pc_range_batch."""
import ctypes as C

import numpy as np
import pytest

import oracle
from knn_brute import brute_knn
from pointcloudtraj_b200 import (PC_DEVICE, PC_HOST, PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED, PcError,
                                 PointCloudIndex, synth)
from pointcloudtraj_b200 import _lib as L

pytestmark = pytest.mark.gpu

PATHS = [PC_QUERY_UNSORTED, PC_QUERY_SORTED]


@pytest.fixture(scope="module")
def ix():
    h = PointCloudIndex(max_points=1 << 18, device=0)
    yield h
    h.close()


def _knn(ix, q, k, r=None, flags=PC_QUERY_AUTO, space=PC_HOST):
    if space == PC_DEVICE:
        import torch
        i, d = ix.knn(torch.from_numpy(np.ascontiguousarray(q)).cuda(), k, r, flags)
        return i.cpu().numpy(), d.cpu().numpy()
    return ix.knn(q, k, r, flags)


def _assert_rows(gi, gd, bi, bd, what=""):
    assert gi.shape == bi.shape, what
    bad = np.nonzero((gi != bi).any(1) | (gd != bd.astype(np.float32)).any(1))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} rows differ, first {bad[:5]}: gpu {gi[bad[0]]} {gd[bad[0]]} brute {bi[bad[0]]} {bd[bad[0]]}"


def _forest_queries(pts, half, seed):
    rng = np.random.default_rng(seed)
    inside = synth.rrt_queries(400, half, seed=seed, lattice_frac=0.5)
    near = pts[rng.integers(0, len(pts), 400)] + rng.normal(0, 0.05, (400, 3)).astype(np.float32)
    far = synth.rrt_queries(100, half, seed=seed + 1) + np.float32(3 * half)
    return np.ascontiguousarray(np.concatenate([inside, near, far]).astype(np.float32))


@pytest.mark.parametrize("variant", ["J", "L"])
def test_knn_forest_200k(ix, variant):
    pts, half = synth.forest_cloud(200_000, seed=11, variant=variant, return_half=True)
    q = _forest_queries(pts, half, 3)
    ix.build(pts)
    for r in (None, 0.3):
        bi, bd = brute_knn(pts, q, 32, r)         # the rows of every k <= 32 are prefixes of these
        for k in (2, 4, 16, 32):
            for flags in PATHS:
                for space in (PC_HOST, PC_DEVICE):
                    gi, gd = _knn(ix, q, k, r, flags, space)
                    _assert_rows(gi, gd, bi[:, :k], bd[:, :k], f"{variant} k={k} r={r} flags={flags} space={space}")


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 9, 33, 65, 4097])
def test_knn_tree_shapes(ix, n):
    rng = np.random.default_rng(n)
    pts = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
    q = np.concatenate([rng.uniform(-3, 3, (200, 3)), pts[: min(n, 50)]]).astype(np.float32)
    ix.build(pts)
    for r in (None, 1.0):
        bi, bd = brute_knn(pts, q, 32, r)
        for flags in PATHS:
            for space in (PC_HOST, PC_DEVICE):
                gi, gd = _knn(ix, q, 32, r, flags, space)
                _assert_rows(gi, gd, bi, bd, f"n={n} r={r} flags={flags} space={space}")
                for row in gi:
                    real = row[row >= 0]
                    assert len(np.unique(real)) == len(real), "a point appears twice in a row"


def test_knn_degenerate_clouds(ix):
    # all points coincident: indices 0..k-1, all distances equal
    pts = np.tile(np.array([[1.0, 2.0, 3.0]], np.float32), (100, 1))
    q = np.array([[1.0, 2.0, 3.0], [0.0, 0.0, 0.0], [5.0, -1.0, 2.5]], np.float32)
    ix.build(pts)
    for flags in PATHS:
        gi, gd = _knn(ix, q, 32, None, flags)
        assert (gi == np.arange(32)).all() and (gd == gd[:, :1]).all()
    # every point twice, queries on points (d2 = 0 first)
    rng = np.random.default_rng(7)
    base = rng.uniform(-1, 1, (500, 3)).astype(np.float32)
    pts = np.concatenate([base, base])
    q = np.concatenate([base[:100], rng.uniform(-1, 1, (100, 3)).astype(np.float32)])
    ix.build(pts)
    bi, bd = brute_knn(pts, q, 8)
    for flags in PATHS:
        for space in (PC_HOST, PC_DEVICE):
            gi, gd = _knn(ix, q, 8, None, flags, space)
            _assert_rows(gi, gd, bi, bd, f"duplicates flags={flags} space={space}")
            assert (gd[:100, :2] == 0).all() and (gi[:100, 0] == np.arange(100)).all() and (gi[:100, 1] == np.arange(500, 600)).all()
    # q_stride 4 (pcl::PointXYZ layout)
    q4 = np.concatenate([q, np.full((len(q), 1), 77.0, np.float32)], 1)
    for flags in PATHS:
        gi, gd = _knn(ix, q4, 8, 0.5, flags)
        bi, bd = brute_knn(pts, q, 8, 0.5)
        _assert_rows(gi, gd, bi, bd, f"stride 4 flags={flags}")
    # empty index: padding only; empty batch
    ix.build(np.zeros((0, 3), np.float32))
    for flags in PATHS:
        for space in (PC_HOST, PC_DEVICE):
            gi, gd = _knn(ix, q, 5, None, flags, space)
            assert (gi == -1).all() and np.isinf(gd).all()
    ix.build(base)
    for space in (PC_HOST, PC_DEVICE):
        gi, gd = _knn(ix, np.zeros((0, 3), np.float32), 4, None, PC_QUERY_AUTO, space)
        assert gi.shape == (0, 4) and gd.shape == (0, 4)


def test_knn_matches_nearest(ix):
    pts, half = synth.forest_cloud(100_000, seed=5, variant="L", return_half=True)
    q = synth.rrt_queries(20_000, half, seed=9, lattice_frac=0.5)
    ix.build(pts)
    ni, nd = ix.nearest(q)
    for flags in (PC_QUERY_AUTO,) + tuple(PATHS):
        gi, gd = ix.knn(q, 1, None, flags)            # k = 1 unbounded is pc_nearest_batch
        assert (gi[:, 0] == ni).all() and (gd[:, 0] == nd).all()
        for k in (2, 8, 32):                          # the kNN kernels' first column
            gi, gd = ix.knn(q, k, None, flags)
            assert (gi[:, 0] == ni).all() and (gd[:, 0] == nd).all(), (k, flags)
        gi, gd = ix.knn(q, 1, 100.0, flags)           # bounded k = 1 runs the kNN kernels
        assert (gi[:, 0] == ni).all() and (gd[:, 0] == nd).all()


def test_knn_bounded_matches_range(ix):
    pts, half = synth.forest_cloud(100_000, seed=8, variant="L", return_half=True)
    q = synth.rrt_queries(3000, half, seed=4, lattice_frac=0.5)
    ix.build(pts)
    r = 0.35
    off, lst = ix.range(q, r)
    for k in (3, 32):
        for flags in PATHS:
            gi, gd = ix.knn(q, k, r, flags)
            for j in range(len(q)):
                ids = lst[off[j]:off[j + 1]].astype(np.int64)
                s = oracle.pair_d2(pts, np.repeat(q[j:j + 1], len(ids), 0), ids)
                o = np.lexsort((ids, s))[:k]
                assert gi[j, : len(o)].tolist() == ids[o].tolist(), (k, flags, j)
                assert (gd[j, : len(o)] == s[o].astype(np.float32)).all()
                assert (gi[j, len(o):] == -1).all() and np.isinf(gd[j, len(o):]).all()


def test_knn_scale_2m_queries():
    pts, half = synth.forest_cloud(1_000_000, variant="J", return_half=True)
    q = synth.rrt_queries(2_000_000, half, seed=1)
    with PointCloudIndex(max_points=len(pts), device=0) as h:
        h.build(pts)
        si, sd = h.knn(q, 8, None, PC_QUERY_SORTED)
        ui, ud = h.knn(q, 8, None, PC_QUERY_UNSORTED)
        ai, ad = h.knn(q, 8, None, PC_QUERY_AUTO)
        assert (si == ui).all() and (sd == ud).all() and (ai == si).all() and (ad == sd).all()
        sub = np.random.default_rng(0).choice(len(q), 5000, replace=False)
        bi, bd = brute_knn(pts, q[sub], 8)
        _assert_rows(si[sub], sd[sub], bi, bd, "2M sub-sample")


def test_knn_incoherent_packets(ix):
    a, half = synth.forest_cloud(20_000, seed=2, variant="J", return_half=True)
    b = a + np.array([150.0, 0.0, 0.0], np.float32)
    pts = np.concatenate([a, b])
    qa = synth.rrt_queries(20_000, half, seed=3)
    qb = synth.rrt_queries(20_000, half, seed=4) + np.array([150.0, 0.0, 0.0], np.float32)
    q = np.empty((40_000, 3), np.float32)
    q[0::2], q[1::2] = qa, qb
    ix.build(pts)
    sub = np.arange(0, len(q), 7)
    for r in (None, 0.5):
        gi, gd = _knn(ix, q, 16, r, PC_QUERY_SORTED, PC_DEVICE)
        bi, bd = brute_knn(pts, q[sub], 16, r)
        _assert_rows(gi[sub], gd[sub], bi, bd, f"two clusters r={r}")
        ui, ud = _knn(ix, q, 16, r, PC_QUERY_UNSORTED, PC_HOST)
        assert (ui == gi).all() and (ud == gd).all()


def test_knn_refusals(ix):
    ix.build(synth.uniform_cloud(1000))
    q = np.zeros((4, 3), np.float32)
    for k in (0, 33):
        with pytest.raises(PcError) as e:
            ix.knn(q, k)
        assert e.value.code == L.PC_EINVAL
    lib = L.load()
    oi = np.empty(4 * 4, np.int32)
    od = np.empty(4 * 4, np.float32)
    for space, k in ((L.PC_HOST_ASYNC, 4), (L.PC_DEVICE_ASYNC, 4), (7, 4), (L.PC_HOST, -1)):
        rc = lib.pc_knn_batch(ix._h, C.c_void_p(q.ctypes.data), 4, 3, space, 0, k, -1.0, C.c_void_p(oi.ctypes.data), C.c_void_p(od.ctypes.data))
        assert rc == L.PC_EINVAL
    with pytest.raises(PcError):
        ix.knn(q, 4, float("nan"))
    with PointCloudIndex(max_points=1000, device=0) as h:
        h.build(synth.uniform_cloud(1000))
        h.batch_shard(0, 2)
        with pytest.raises(PcError) as e:
            h.knn(q, 4)
        assert e.value.code == L.PC_EINVAL
        with pytest.raises(PcError):
            h.knn(q, 1)                               # k = 1 too: no rows are left unwritten
