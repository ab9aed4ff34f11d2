"""GPU tests of pc_segment_nearest_batch: bit-equal with the fp64 brute force (tests/segment_brute.c) under every flag and in both
memory spaces, on forests, tree shapes, lattices with exact ties, points at float-ulp distance from long segments, map-crossing
and far-away segments; plus its exact relations to pc_nearest_batch and pc_knn_batch, polylines, and the refusals."""
import ctypes as C
import os

import numpy as np
import pytest

from pointcloudtraj_b200 import (PC_DEVICE, PC_HOST, PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED, PcError,
                                 PointCloudIndex, synth)
from pointcloudtraj_b200 import _lib as L
from segment_brute import brute_segment

pytestmark = pytest.mark.gpu

FLAGS = [PC_QUERY_AUTO, PC_QUERY_UNSORTED, PC_QUERY_SORTED]
SPACES = [PC_HOST, PC_DEVICE]


@pytest.fixture(scope="module")
def ix():
    h = PointCloudIndex(max_points=1 << 20, device=0)
    yield h
    h.close()


def _seg(ix, a, b, r=None, flags=PC_QUERY_AUTO, space=PC_HOST):
    if space == PC_DEVICE:
        import torch
        i, d = ix.segment_nearest(torch.from_numpy(np.ascontiguousarray(a)).cuda(), torch.from_numpy(np.ascontiguousarray(b)).cuda(), r, flags)
        return i.cpu().numpy(), d.cpu().numpy()
    return ix.segment_nearest(a, b, r, flags)


def _assert_same(gi, gd, bi, bd, what=""):
    bad = np.nonzero((gi != bi) | (gd.view(np.uint32) != bd.astype(np.float32).view(np.uint32)))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} rows differ, first {bad[:5]}: gpu {gi[bad[0]]} {gd[bad[0]]} brute {bi[bad[0]]} {bd[bad[0]]}"


def _check_all(ix, pts, a, b, ranges, what, flags_list=FLAGS, spaces=SPACES):
    for r in ranges:
        bi, bd = brute_segment(pts, a, b, r)
        for flags in flags_list:
            for space in spaces:
                gi, gd = _seg(ix, a, b, r, flags, space)
                _assert_same(gi, gd, bi, bd, f"{what} r={r} flags={flags} space={space}")


def _random_segments(rng, starts, lengths):
    d = rng.normal(size=(len(starts), 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return starts.astype(np.float32), (starts + d * np.asarray(lengths)[:, None]).astype(np.float32)


@pytest.mark.parametrize("variant", ["J", "L"])
def test_segment_forest_200k(ix, variant):
    pts, half = synth.forest_cloud(200_000, seed=11, variant=variant, return_half=True)
    ix.build(pts)
    rng = np.random.default_rng(5)
    n = 900
    starts = np.concatenate([synth.rrt_queries(600, half, seed=3, lattice_frac=0.5),
                             pts[rng.integers(0, len(pts), 300)] + rng.normal(0, 0.05, (300, 3)).astype(np.float32)])
    lengths = rng.choice([0.0, 0.05, 0.3, 1.0, 4.0, 15.0, 50.0], n) * rng.uniform(0.5, 1.0, n)
    lengths[:50] = 0.0
    a, b = _random_segments(rng, starts, lengths)
    _check_all(ix, pts, a, b, (None, 0.5, 2.0), f"forest {variant}")


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 33, 64, 65, 1023, 1024, 1025, 4097])
def test_segment_tree_shapes(ix, n):
    rng = np.random.default_rng(n)
    pts = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
    a = np.concatenate([rng.uniform(-3, 3, (200, 3)), pts[: min(n, 50)]]).astype(np.float32)
    b = (a + rng.normal(0, 1.5, a.shape)).astype(np.float32)
    b[-min(n, 50) // 2:] = a[-min(n, 50) // 2:]
    ix.build(pts)
    _check_all(ix, pts, a, b, (None, 1.0), f"n={n}", flags_list=[PC_QUERY_UNSORTED, PC_QUERY_SORTED])


def test_segment_lattice_ties(ix):
    # every lattice point twice; segments along lattice lines and through lattice points: d2 = 0 and exact ties everywhere
    g = np.arange(16, dtype=np.float32) * 0.25
    base = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    rng = np.random.default_rng(9)
    pts = np.concatenate([base, base[rng.permutation(len(base))]]).astype(np.float32)
    ix.build(pts)
    i0 = rng.integers(0, len(base), 400)
    i1 = rng.integers(0, len(base), 400)
    a = base[i0].copy()
    b = base[i1].copy()
    ax = rng.integers(0, 3, 200)
    b[:200] = a[:200]
    b[np.arange(200), ax] = base[i1[:200], ax]                      # along a lattice line
    off = np.concatenate([a[:100] + 0.125, a[100:200] - 0.125])     # between lattice lines, equidistant from several points
    a2, b2 = off.astype(np.float32), (off + np.array([1.0, 0.5, 0.0], np.float32)).astype(np.float32)
    A, B = np.concatenate([a, a2]), np.concatenate([b, b2])
    _check_all(ix, pts, A, B, (None, 0.125, 0.3), "lattice")


def test_segment_ulp_distance(ix):
    # long segments whose nearest points lie far from A, with cloud points a few float ulps off the segment: the best d2 is
    # near 0, where the fp64 expression's error is absolute (the tau term of the node test)
    rng = np.random.default_rng(21)
    a = rng.uniform(-40, 40, (64, 3)).astype(np.float32)
    b = (a + rng.normal(0, 30, (64, 3))).astype(np.float32)
    t = rng.uniform(0.2, 0.95, (64, 40))
    on = a[:, None, :].astype(np.float64) + t[..., None] * (b - a)[:, None, :].astype(np.float64)
    p = on.astype(np.float32)
    ulps = rng.integers(-3, 4, p.shape).astype(np.int32)
    p = (p.view(np.int32) + ulps).view(np.float32)                  # nudged by up to 3 ulps per coordinate
    pts = np.concatenate([p.reshape(-1, 3), rng.uniform(-80, 80, (20000, 3)).astype(np.float32)])
    ix.build(pts)
    _check_all(ix, pts, a, b, (None, 1e-3), "ulp")
    # the same with the segments reversed (the fp64 expression is not symmetric in a and b)
    _check_all(ix, pts, b, a, (None,), "ulp reversed")


def test_segment_crossing_and_far(ix):
    pts, half = synth.forest_cloud(200_000, seed=2, variant="J", return_half=True)
    ix.build(pts)
    lo, hi = pts.min(0), pts.max(0)
    rng = np.random.default_rng(3)
    # corner to corner and wall to wall: the frontier fills up and falls back to depth-first steps
    a = np.array([lo, [lo[0], hi[1], lo[2]], [lo[0], 0, 1.0], [0, lo[1], 2.0]], np.float32)
    b = np.array([hi, [hi[0], lo[1], hi[2]], [hi[0], 0, 1.0], [0, hi[1], 2.0]], np.float32)
    a = np.concatenate([a, rng.uniform(lo, hi, (40, 3))]).astype(np.float32)
    b = np.concatenate([b, rng.uniform(lo, hi, (40, 3))]).astype(np.float32)
    _check_all(ix, pts, a, b, (None, 0.5), "crossing")
    # endpoints at 1e6 m, the cloud at the origin and the cloud moved there too
    fa = np.array([[1e6, 0, 0], [0, 1e6, 3], [1e6, 1e6, 1e6], [-1e6, 5, 1]], np.float32)
    fb = np.array([[-1e6, 0, 1], [0, 1e6 + 40, 3], [1e6, 1e6, 1e6], [1e6, -5, 2]], np.float32)
    _check_all(ix, pts, fa, fb, (None, 1e6), "far")
    shifted = (pts.astype(np.float64) + 1e6).astype(np.float32)
    ix.build(shifted)
    sa = (a.astype(np.float64) + 1e6).astype(np.float32)
    sb = (b.astype(np.float64) + 1e6).astype(np.float32)
    _check_all(ix, shifted, sa, sb, (None, 0.5), "shifted to 1e6")


def test_segment_nonfinite_empty_and_sizes(ix):
    rng = np.random.default_rng(1)
    pts = rng.uniform(-5, 5, (5000, 3)).astype(np.float32)
    a = rng.uniform(-5, 5, (12, 3)).astype(np.float32)
    b = rng.uniform(-5, 5, (12, 3)).astype(np.float32)
    bad = [np.nan, np.inf, -np.inf]
    for j in range(9):
        (a if j % 2 == 0 else b)[j, j % 3] = bad[j % 3]
    for cloud in (pts, pts[:0]):
        ix.build(cloud)
        for flags in FLAGS:
            for space in SPACES:
                for r in (None, 1.0):
                    gi, gd = _seg(ix, a, b, r, flags, space)
                    assert (gi[:9] == -1).all() and np.isnan(gd[:9]).all(), (flags, space, r, gi, gd)
                    if len(cloud) == 0:
                        assert (gi[9:] == -1).all() and np.isinf(gd[9:]).all()
        if len(cloud):
            bi, bd = brute_segment(cloud, a, b)
            _assert_same(*_seg(ix, a, b), bi, bd, "finite rows")
    ix.build(pts)
    for m in (0, 1):
        for space in SPACES:
            gi, gd = _seg(ix, a[9:9 + m], b[9:9 + m], None, PC_QUERY_AUTO, space)
            assert len(gi) == m and len(gd) == m
            if m:
                bi, bd = brute_segment(pts, a[9:10], b[9:10])
                _assert_same(gi, gd, bi, bd, "m = 1")


def _raw(ix, pa, pb, m, stride, space, flags=PC_QUERY_AUTO, r=-1.0):
    """pc_segment_nearest_batch on raw addresses (host numpy / device torch), returns (rc, idx, d2)."""
    if space == PC_DEVICE:
        import torch
        oi = torch.empty(max(m, 1), dtype=torch.int32, device="cuda")
        od = torch.empty(max(m, 1), dtype=torch.float32, device="cuda")
        rc = ix._L.pc_segment_nearest_batch(ix._h, C.c_void_p(pa), C.c_void_p(pb), m, stride, space, flags, r,
                                            C.c_void_p(oi.data_ptr()), C.c_void_p(od.data_ptr()))
        torch.cuda.synchronize()
        ix.sync()
        return rc, oi.cpu().numpy()[:m], od.cpu().numpy()[:m]
    oi = np.empty(max(m, 1), np.int32)
    od = np.empty(max(m, 1), np.float32)
    rc = ix._L.pc_segment_nearest_batch(ix._h, C.c_void_p(pa), C.c_void_p(pb), m, stride, space, flags, r,
                                        C.c_void_p(oi.ctypes.data), C.c_void_p(od.ctypes.data))
    return rc, oi[:m], od[:m]


def test_segment_stride_and_polyline(ix):
    pts, half = synth.forest_cloud(200_000, seed=7, variant="L", return_half=True)
    ix.build(pts)
    rng = np.random.default_rng(8)
    # a random-walk polyline of 3001 points through the map: 3000 segments, b = a + stride
    steps = rng.normal(0, 0.4, (3001, 3)).astype(np.float32)
    poly = (np.cumsum(steps, 0) * np.float32(0.3) + np.array([0, 0, 1.5], np.float32)).astype(np.float32)
    bi, bd = brute_segment(pts, poly[:-1], poly[1:])
    bi_r, bd_r = brute_segment(pts, poly[:-1], poly[1:], 0.5)
    for stride in (3, 4):
        arr = np.zeros((len(poly), stride), np.float32)
        arr[:, :3] = poly
        if stride == 4:
            arr[:, 3] = np.nan                                       # the pad word is never read
        import torch
        dev = torch.from_numpy(arr).cuda()
        for space in SPACES:
            base = arr.ctypes.data if space == PC_HOST else dev.data_ptr()
            for flags in FLAGS:
                for r, (ei, ed) in ((-1.0, (bi, bd)), (0.5, (bi_r, bd_r))):
                    rc, gi, gd = _raw(ix, base, base + 4 * stride, len(poly) - 1, stride, space, flags, r)
                    assert rc == L.PC_OK
                    _assert_same(gi, gd, ei, ed, f"polyline stride={stride} space={space} flags={flags} r={r}")
        # two separate arrays of that stride through the wrapper
        a4, b4 = arr[:-1].copy(), arr[1:].copy()
        for space in SPACES:
            gi, gd = _seg(ix, a4, b4, None, PC_QUERY_SORTED, space)
            _assert_same(gi, gd, bi, bd, f"stride={stride} arrays space={space}")


def test_segment_multi_chunk_host():
    os.environ["PC_HOST_CHUNK_QUERIES"] = "4096"
    try:
        h = PointCloudIndex(max_points=1 << 18, device=0)
    finally:
        del os.environ["PC_HOST_CHUNK_QUERIES"]
    pts, half = synth.forest_cloud(200_000, seed=4, variant="J", return_half=True)
    h.build(pts)
    rng = np.random.default_rng(2)
    starts = synth.rrt_queries(20_000, half, seed=6)
    a, b = _random_segments(rng, starts, rng.uniform(0, 3, 20_000))
    bi, bd = brute_segment(pts, a, b)
    for flags in FLAGS:
        gi, gd = h.segment_nearest(a, b, None, flags)
        _assert_same(gi, gd, bi, bd, f"multi-chunk flags={flags}")
    # a polyline across chunk boundaries
    rc, gi, gd = _raw(h, starts.ctypes.data, starts.ctypes.data + 12, len(starts) - 1, 3, PC_HOST)
    ei, ed = brute_segment(pts, starts[:-1], starts[1:])
    assert rc == L.PC_OK
    _assert_same(gi, gd, ei, ed, "multi-chunk polyline")
    h.close()


def test_segment_1m_batch(ix):
    pts, half = synth.forest_cloud(200_000, seed=12, variant="J", return_half=True)
    ix.build(pts)
    rng = np.random.default_rng(13)
    m = 1_000_000
    starts = synth.rrt_queries(m, half, seed=14)
    a, b = _random_segments(rng, starts, rng.choice([0.0, 0.1, 1.0, 10.0], m))
    rows = rng.choice(m, 3000, replace=False)
    for r in (None, 0.5):
        bi, bd = brute_segment(pts, a[rows], b[rows], r)
        ref = None
        for flags in FLAGS:
            for space in SPACES:
                gi, gd = _seg(ix, a, b, r, flags, space)
                _assert_same(gi[rows], gd[rows], bi, bd, f"1M r={r} flags={flags} space={space}")
                if ref is None:
                    ref = (gi, gd)
                assert (gi == ref[0]).all() and (gd.view(np.uint32) == ref[1].view(np.uint32)).all(), \
                    f"1M r={r}: flags={flags} space={space} differ from the first path"


def test_segment_relations(ix):
    pts, half = synth.forest_cloud(200_000, seed=11, variant="J", return_half=True)
    ix.build(pts)
    q = synth.rrt_queries(50_000, half, seed=15)
    ni, nd = ix.nearest(q)
    for flags in FLAGS:
        for space in SPACES:
            gi, gd = _seg(ix, q, q, None, flags, space)
            assert (gi == ni).all() and (gd.view(np.uint32) == nd.view(np.uint32)).all(), f"degenerate != nearest ({flags}, {space})"
            for r in (0.3, 1.0):
                ki, kd = ix.knn(q, 1, r)
                gi, gd = _seg(ix, q, q, r, flags, space)
                assert (gi == ki[:, 0]).all() and (gd.view(np.uint32) == kd[:, 0].view(np.uint32)).all(), f"bounded degenerate != knn ({r})"


def test_segment_sampling_gap(ix):
    # one obstacle point midway between two samples: both endpoint queries report a clearance above r, the segment does not
    r = 0.5
    a = np.array([[0.0, 0.0, 1.0]], np.float32)
    b = np.array([[2.0, 0.0, 1.0]], np.float32)
    p = np.array([[1.0, 0.45, 1.0], [-3.0, 0.0, 1.0], [5.0, 0.0, 1.0]], np.float32)
    ix.build(p)
    _, da = ix.nearest(a)
    _, db = ix.nearest(b)
    assert da[0] > r * r and db[0] > r * r
    bi, bd = brute_segment(p, a, b)
    assert bi[0] == 0 and bd[0] <= r * r
    for flags in FLAGS:
        for space in SPACES:
            for rr in (None, r):
                gi, gd = _seg(ix, a, b, rr, flags, space)
                _assert_same(gi, gd, bi, bd, f"sampling gap r={rr} flags={flags} space={space}")


def test_segment_refusals(ix):
    ix.build(np.zeros((10, 3), np.float32))
    a = np.zeros((4, 3), np.float32)
    pa = a.ctypes.data
    f = ix._L.pc_segment_nearest_batch
    out_i = np.empty(4, np.int32)
    pi = C.c_void_p(out_i.ctypes.data)
    cases = [
        (pa, pa, 4, 5, PC_HOST, 0, -1.0),          # bad stride
        (None, pa, 4, 3, PC_HOST, 0, -1.0),        # NULL a
        (pa, None, 4, 3, PC_HOST, 0, -1.0),        # NULL b
        (pa, pa, 4, 3, L.PC_HOST_ASYNC, 0, -1.0),
        (pa, pa, 4, 3, L.PC_DEVICE_ASYNC, 0, -1.0),
        (pa, pa, 4, 3, PC_HOST, 1, -1.0),          # unknown flags
        (pa, pa, 4, 3, PC_HOST, 8, -1.0),
        (pa, pa, 4, 3, PC_HOST, 0, float("nan")),  # NaN range
    ]
    for c in cases:
        rc = f(ix._h, C.c_void_p(c[0]) if c[0] else None, C.c_void_p(c[1]) if c[1] else None, c[2], c[3], c[4], c[5], c[6], pi, None)
        assert rc == L.PC_EINVAL, c
        assert b"pc_segment_nearest_batch" in ix._L.pc_last_error(ix._h), c
    assert f(ix._h, None, None, 0, 3, PC_HOST, 0, -1.0, None, None) == L.PC_OK          # m = 0, NULL arrays
    ix.batch_shard(0, 2)
    try:
        assert f(ix._h, C.c_void_p(pa), C.c_void_p(pa), 4, 3, PC_HOST, 0, -1.0, pi, None) == L.PC_EINVAL
        assert b"pc_segment_nearest_batch" in ix._L.pc_last_error(ix._h)
        with pytest.raises(PcError):
            ix.segment_nearest(a, a)
    finally:
        ix.batch_shard(0, 1)
