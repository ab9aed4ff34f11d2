"""GPU tests of pc_knn_large_batch (k up to 1024): bit-equal with the fp64 brute force (tests/knn_brute.c) under every flag
and in both memory spaces, plus its exact relations to pc_knn_batch and pc_range_sorted_batch."""
import ctypes as C
import os

import numpy as np
import pytest

from knn_brute import brute_knn
from pointcloudtraj_b200 import (PC_DEVICE, PC_HOST, PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED, PcError,
                                 PointCloudIndex, synth)
from pointcloudtraj_b200 import _lib as L
from test_knn_gpu import _assert_rows, _forest_queries

pytestmark = pytest.mark.gpu

FLAGS = [PC_QUERY_AUTO, PC_QUERY_UNSORTED, PC_QUERY_SORTED]
PATHS = [PC_QUERY_UNSORTED, PC_QUERY_SORTED]


@pytest.fixture(scope="module")
def ix():
    h = PointCloudIndex(max_points=1 << 18, device=0)
    yield h
    h.close()


def _knn(ix, q, k, r=None, flags=PC_QUERY_AUTO, space=PC_HOST):
    if space == PC_DEVICE:
        import torch
        i, d = ix.knn_large(torch.from_numpy(np.ascontiguousarray(q)).cuda(), k, r, flags)
        return i.cpu().numpy(), d.cpu().numpy()
    return ix.knn_large(q, k, r, flags)


@pytest.mark.parametrize("variant", ["J", "L"])
def test_knn_large_forest_200k(ix, variant):
    pts, half = synth.forest_cloud(200_000, seed=11, variant=variant, return_half=True)
    q = _forest_queries(pts, half, 3)
    ix.build(pts)
    for r in (None, 0.3, 1.0):
        bi, bd = brute_knn(pts, q, 1024, r)       # the rows of every k <= 1024 are prefixes of these
        for k in (33, 64, 100, 256, 1024):
            for flags in FLAGS:
                for space in (PC_HOST, PC_DEVICE):
                    gi, gd = _knn(ix, q, k, r, flags, space)
                    _assert_rows(gi, gd, bi[:, :k], bd[:, :k], f"{variant} k={k} r={r} flags={flags} space={space}")


@pytest.mark.parametrize("n", [1, 2, 5, 33, 64, 65, 1023, 1024, 1025, 4097])
def test_knn_large_tree_shapes(ix, n):
    rng = np.random.default_rng(n)
    pts = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
    q = np.concatenate([rng.uniform(-3, 3, (200, 3)), pts[: min(n, 50)]]).astype(np.float32)
    ix.build(pts)
    for r in (None, 1.0):
        bi, bd = brute_knn(pts, q, 1024, r)
        for k in (33, 1024):
            for flags in PATHS:
                for space in (PC_HOST, PC_DEVICE):
                    gi, gd = _knn(ix, q, k, r, flags, space)
                    _assert_rows(gi, gd, bi[:, :k], bd[:, :k], f"n={n} k={k} r={r} flags={flags} space={space}")
                    for row in gi:
                        real = row[row >= 0]
                        assert len(np.unique(real)) == len(real), "a point appears twice in a row"


def test_knn_large_ties(ix):
    # 2000 identical points: every distance equal, the row is 0..k-1 (equal keys cross many queue flushes)
    pts = np.tile(np.array([[1.0, 2.0, 3.0]], np.float32), (2000, 1))
    q = np.array([[1.0, 2.0, 3.0], [0.0, 0.0, 0.0], [5.0, -1.0, 2.5]], np.float32)
    ix.build(pts)
    for k in (100, 1024):
        for flags in FLAGS:
            for space in (PC_HOST, PC_DEVICE):
                gi, gd = _knn(ix, q, k, None, flags, space)
                assert (gi == np.arange(k)).all() and (gd == gd[:, :1]).all(), (k, flags, space)
    # a lattice with every point three times: long runs of equal distances at every k
    rng = np.random.default_rng(7)
    base = (rng.integers(0, 12, size=(1500, 3)) * 0.25).astype(np.float32)
    pts = np.concatenate([base, base, base])
    q = np.concatenate([base[:100], (rng.integers(0, 23, size=(100, 3)) * 0.125)]).astype(np.float32)
    ix.build(pts)
    for r in (None, 0.6):
        bi, bd = brute_knn(pts, q, 1024, r)
        for k in (33, 257, 1024):
            for flags in PATHS:
                for space in (PC_HOST, PC_DEVICE):
                    gi, gd = _knn(ix, q, k, r, flags, space)
                    _assert_rows(gi, gd, bi[:, :k], bd[:, :k], f"lattice k={k} r={r} flags={flags} space={space}")


def test_knn_large_relations(ix):
    pts, half = synth.forest_cloud(100_000, seed=5, variant="L", return_half=True)
    q = synth.rrt_queries(5000, half, seed=9, lattice_frac=0.5)
    ix.build(pts)
    for r in (None, 0.8):
        rows = {}
        for k in (33, 64, 200, 1024):
            gi, gd = ix.knn_large(q, k, r)
            for flags in PATHS:                                        # 4. every flag gives the same rows
                fi, fd = ix.knn_large(q, k, r, flags)
                assert (fi == gi).all() and (fd == gd).all(), (k, r, flags)
            rows[k] = gi, gd
        si, sd = ix.knn(q, 32, r)                                      # 1. the first 32 columns are pc_knn_batch's row
        for k, (gi, gd) in rows.items():
            assert (gi[:, :32] == si).all() and (gd[:, :32] == sd).all(), (k, r)
        for k1, k2 in ((33, 64), (64, 200), (200, 1024)):             # 2. a shorter row is a prefix of a longer one
            assert (rows[k1][0] == rows[k2][0][:, :k1]).all() and (rows[k1][1] == rows[k2][1][:, :k1]).all(), (k1, k2, r)
        if r is None:
            continue
        for k, (gi, gd) in rows.items():                               # 3. bounded rows are pc_range_sorted_batch's
            off, ri, rd = ix.range_sorted(q, r, max_nn=k)
            n = np.diff(off)
            mask = np.arange(k)[None, :] < n[:, None]
            assert (gi[mask] == ri).all() and (gd[mask] == rd).all(), k
            assert (gi[~mask] == -1).all() and np.isinf(gd[~mask]).all(), k
    for k in (1, 8, 32):                                               # k <= 32 is pc_knn_batch
        for r in (None, 0.8):
            gi, gd = ix.knn_large(q, k, r)
            si, sd = ix.knn(q, k, r)
            assert (gi == si).all() and (gd == sd).all(), (k, r)


def test_knn_large_degenerate(ix):
    rng = np.random.default_rng(4)
    pts = rng.uniform(-1, 1, (3000, 3)).astype(np.float32)
    q = rng.uniform(-1.2, 1.2, (150, 3)).astype(np.float32)
    # q_stride 4 (pcl::PointXYZ layout)
    ix.build(pts)
    q4 = np.concatenate([q, np.full((len(q), 1), 77.0, np.float32)], 1)
    bi, bd = brute_knn(pts, q, 300, 0.5)
    for flags in PATHS:
        for space in (PC_HOST, PC_DEVICE):
            gi, gd = _knn(ix, q4, 300, 0.5, flags, space)
            _assert_rows(gi, gd, bi, bd, f"stride 4 flags={flags} space={space}")
    # empty batch
    for space in (PC_HOST, PC_DEVICE):
        gi, gd = _knn(ix, np.zeros((0, 3), np.float32), 64, None, PC_QUERY_AUTO, space)
        assert gi.shape == (0, 64) and gd.shape == (0, 64)
    # empty index: padding only
    ix.build(np.zeros((0, 3), np.float32))
    for flags in FLAGS:
        for space in (PC_HOST, PC_DEVICE):
            gi, gd = _knn(ix, q, 64, None, flags, space)
            assert (gi == -1).all() and np.isinf(gd).all()


def test_knn_large_host_chunks():
    # PC_HOST_CHUNK_QUERIES = 1024 gives chunks of 1024 * 32 / k queries: 32 at k = 1024, so 40 chunks over the lanes
    rng = np.random.default_rng(12)
    pts = rng.uniform(-3, 3, (50_000, 3)).astype(np.float32)
    q = rng.uniform(-3.5, 3.5, (1280, 3)).astype(np.float32)
    os.environ["PC_HOST_CHUNK_QUERIES"] = "1024"
    try:
        h = PointCloudIndex(max_points=len(pts), device=0)
    finally:
        del os.environ["PC_HOST_CHUNK_QUERIES"]
    with h:
        h.build(pts)
        for k, r in ((1024, None), (100, 0.7)):
            bi, bd = brute_knn(pts, q, k, r)
            for flags in PATHS:
                gi, gd = h.knn_large(q, k, r, flags)
                _assert_rows(gi, gd, bi, bd, f"chunked k={k} r={r} flags={flags}")


def test_knn_large_scale_1m_queries():
    pts, half = synth.forest_cloud(1_000_000, variant="J", return_half=True)
    q = synth.rrt_queries(1_000_000, half, seed=1)
    with PointCloudIndex(max_points=len(pts), device=0) as h:
        h.build(pts)
        si, sd = h.knn_large(q, 64, None, PC_QUERY_SORTED)
        ui, ud = h.knn_large(q, 64, None, PC_QUERY_UNSORTED)
        assert (si == ui).all() and (sd == ud).all()
        del ui, ud
        ai, ad = h.knn_large(q, 64, None, PC_QUERY_AUTO)
        assert (ai == si).all() and (ad == sd).all()
        del ai, ad
        sub = np.random.default_rng(0).choice(len(q), 2000, replace=False)
        bi, bd = brute_knn(pts, q[sub], 64)
        _assert_rows(si[sub], sd[sub], bi, bd, "1M sub-sample")


def test_knn_large_refusals(ix):
    ix.build(synth.uniform_cloud(1000))
    q = np.zeros((4, 3), np.float32)
    lib = L.load()
    oi = np.empty(4 * 1100, np.int32)
    od = np.empty(4 * 1100, np.float32)
    call = lambda space, flags, k, r: lib.pc_knn_large_batch(ix._h, C.c_void_p(q.ctypes.data), 4, 3, space, flags, k, r,
                                                             C.c_void_p(oi.ctypes.data), C.c_void_p(od.ctypes.data))
    for k in (0, -1, 1025):
        assert call(PC_HOST, 0, k, -1.0) == L.PC_EINVAL, k
    assert "pc_range_sorted_batch" in lib.pc_last_error(ix._h).decode()
    assert call(PC_HOST, 0, 64, float("nan")) == L.PC_EINVAL
    assert call(PC_HOST, 1, 64, -1.0) == L.PC_EINVAL                 # unknown flag bit
    for space in (L.PC_HOST_ASYNC, L.PC_DEVICE_ASYNC, 7):
        assert call(space, 0, 64, -1.0) == L.PC_EINVAL, space
    assert call(PC_HOST, 0, 1024, -1.0) == L.PC_OK
    with pytest.raises(PcError) as e:
        ix.knn_large(q, 1025)
    assert e.value.code == L.PC_EINVAL
    with pytest.raises(PcError) as e:                                 # pc_knn_batch keeps its limit
        ix.knn(q, 33)
    assert e.value.code == L.PC_EINVAL
    with PointCloudIndex(max_points=1000, device=0) as h:
        h.build(synth.uniform_cloud(1000))
        h.batch_shard(0, 2)
        for k in (8, 64):
            with pytest.raises(PcError) as e:
                h.knn_large(q, k)
            assert e.value.code == L.PC_EINVAL
