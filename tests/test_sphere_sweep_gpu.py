"""GPU tests of pc_sphere_sweep_batch: bit-equal with the fp64 brute force (tests/sweep_brute.c, t rounded down to float32
here) under every flag and in both memory spaces, on forests, tree shapes, lattices with exact ties, grazing contacts on long
segments, segments starting inside the cloud, contacts through the B clause, far and non-finite endpoints, polylines and
large batches; plus its exact relations to pc_range_batch, its monotonicity in the radius, the banded agreement with
pc_segment_nearest_batch, and the refusals."""
import ctypes as C
import os

import numpy as np
import pytest

from pointcloudtraj_b200 import (PC_DEVICE, PC_HOST, PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED, PcError,
                                 PointCloudIndex, synth)
from pointcloudtraj_b200 import _lib as L
from segment_brute import brute_segment
from sweep_brute import b_clause_rows, brute_sweep, numpy_quadratic_t, round_down_f32

pytestmark = pytest.mark.gpu

FLAGS = [PC_QUERY_AUTO, PC_QUERY_UNSORTED, PC_QUERY_SORTED]
SPACES = [PC_HOST, PC_DEVICE]


@pytest.fixture(scope="module")
def ix():
    h = PointCloudIndex(max_points=1 << 20, device=0)
    yield h
    h.close()


def _sweep(ix, a, b, r, flags=PC_QUERY_AUTO, space=PC_HOST):
    if space == PC_DEVICE:
        import torch
        i, t = ix.sphere_sweep(torch.from_numpy(np.ascontiguousarray(a)).cuda(), torch.from_numpy(np.ascontiguousarray(b)).cuda(), r, flags)
        return i.cpu().numpy(), t.cpu().numpy()
    return ix.sphere_sweep(a, b, r, flags)


def _assert_same(gi, gt, bi, bt, what=""):
    ft = round_down_f32(bt)
    bad = np.nonzero((gi != bi) | (gt.view(np.uint32) != ft.view(np.uint32)))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} rows differ, first {bad[:5]}: gpu {gi[bad[0]]} {gt[bad[0]]!r} brute {bi[bad[0]]} {bt[bad[0]]!r}"


def _check_all(ix, pts, a, b, radii, what, flags_list=FLAGS, spaces=SPACES):
    for r in radii:
        bi, bt = brute_sweep(pts, a, b, r)
        for flags in flags_list:
            for space in spaces:
                gi, gt = _sweep(ix, a, b, r, flags, space)
                _assert_same(gi, gt, bi, bt, f"{what} r={r} flags={flags} space={space}")


def _random_segments(rng, starts, lengths):
    d = rng.normal(size=(len(starts), 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return starts.astype(np.float32), (starts + d * np.asarray(lengths)[:, None]).astype(np.float32)


@pytest.mark.parametrize("variant", ["J", "L"])
def test_sweep_forest_200k(ix, variant):
    pts, half = synth.forest_cloud(200_000, seed=11, variant=variant, return_half=True)
    ix.build(pts)
    rng = np.random.default_rng(5)
    n = 900
    starts = np.concatenate([synth.rrt_queries(600, half, seed=3, lattice_frac=0.5),
                             pts[rng.integers(0, len(pts), 300)] + rng.normal(0, 0.05, (300, 3)).astype(np.float32)])
    lengths = rng.choice([0.0, 0.05, 0.3, 1.0, 4.0, 15.0, 50.0], n) * rng.uniform(0.5, 1.0, n)
    lengths[:50] = 0.0
    a, b = _random_segments(rng, starts, lengths)
    _check_all(ix, pts, a, b, (0.0, 0.05, 0.5, 2.0), f"forest {variant}")


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 33, 64, 65, 1023, 1024, 1025, 4097])
def test_sweep_tree_shapes(ix, n):
    rng = np.random.default_rng(n)
    pts = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
    a = np.concatenate([rng.uniform(-3, 3, (200, 3)), pts[: min(n, 50)]]).astype(np.float32)
    b = (a + rng.normal(0, 1.5, a.shape)).astype(np.float32)
    b[-min(n, 50) // 2:] = a[-min(n, 50) // 2:]
    ix.build(pts)
    _check_all(ix, pts, a, b, (0.0, 0.3, 1.0), f"n={n}", flags_list=[PC_QUERY_UNSORTED, PC_QUERY_SORTED])


def test_sweep_lattice_ties(ix):
    # every lattice point twice; spheres swept along and across lattice rows: many points touch at exactly equal t
    g = np.arange(16, dtype=np.float32) * 0.25
    base = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    rng = np.random.default_rng(9)
    pts = np.concatenate([base, base[rng.permutation(len(base))]]).astype(np.float32)
    ix.build(pts)
    i0 = rng.integers(0, len(base), 300)
    ax = rng.integers(0, 3, 300)
    a = base[i0].copy()
    a[np.arange(300), ax] = -1.0                                       # outside the lattice, on a lattice line
    b = a.copy()
    b[np.arange(300), ax] = 5.0                                        # along the row: the row's first point and its twin tie
    off = a[:150].copy()
    off[:, (ax[:150] + 1) % 3] += 0.125                                # between two rows: both touch at the same t
    across = base[rng.integers(0, len(base), 150)] + np.float32(0.125)
    A = np.concatenate([a, off, across]).astype(np.float32)
    B = np.concatenate([b, b[:150] + (off - a[:150]), across + np.array([1.0, 0.5, 0.0], np.float32)]).astype(np.float32)
    _check_all(ix, pts, A, B, (0.0, 0.125, 0.25, 0.3), "lattice")
    bi, bt = brute_sweep(pts, A, B, 0.125)
    assert (bi[:300] >= 0).all()


def test_sweep_grazing(ix):
    # points placed laterally at r (1 + k 2^-26) from 30-50 m segments, far from a: the sign of disc flips between neighbours,
    # where the computed t is ill-conditioned (the sqrt(u) term of rho)
    rng = np.random.default_rng(21)
    m = 64
    a = rng.uniform(-40, 40, (m, 3)).astype(np.float32)
    d = rng.normal(size=(m, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    b = (a + d * rng.uniform(30, 50, (m, 1))).astype(np.float32)
    k = np.arange(-12, 13)
    t = rng.uniform(0.4, 0.95, (m, len(k)))
    nrm = np.cross(d[:, None, :], rng.normal(size=(m, len(k), 3)))
    nrm /= np.linalg.norm(nrm, axis=2, keepdims=True)
    clouds = []
    for r in (0.05, 0.5, 2.0):
        p = a[:, None, :] + t[..., None] * (b - a)[:, None, :] + (r * (1 + k * 2.0 ** -26))[None, :, None] * nrm
        clouds.append(p.reshape(-1, 3))
    pts = np.concatenate(clouds + [rng.uniform(-90, 90, (20000, 3))]).astype(np.float32)
    ix.build(pts)
    _check_all(ix, pts, a, b, (0.05, 0.5, 2.0), "grazing")
    _check_all(ix, pts, b, a, (0.5,), "grazing reversed")


def test_sweep_inside_and_b_clause(ix):
    rng = np.random.default_rng(17)
    # contacts that only the B clause reaches (b_clause_rows): one point per segment at exactly r from b
    r = 0.3125
    a, b, p = b_clause_rows(rng, 400, r)
    ix.build(p)
    _check_all(ix, p, a, b, (r,), "B clause")
    bi, bt = brute_sweep(p, a, b, r)
    via_b = [j for j in range(400) if bi[j] == j and bt[j] == 1.0 and numpy_quadratic_t(p[j], a[j], b[j], r) > 1.0]
    assert len(via_b) > 20, "too few contacts through the B clause"
    # segments that start inside the cloud (t = 0) or next to it
    pts, half = synth.forest_cloud(200_000, seed=9, variant="J", return_half=True)
    ix.build(pts)
    s = pts[rng.integers(0, len(pts), 300)] + rng.normal(0, 0.1, (300, 3)).astype(np.float32)
    sa, sb = _random_segments(rng, s, rng.uniform(0, 3, 300))
    _check_all(ix, pts, sa, sb, (0.05, r), "inside")
    assert (brute_sweep(pts, sa, sb, r)[1] == 0).sum() > 50, "too few segments start inside"


def test_sweep_far_nonfinite_empty_and_sizes(ix):
    pts, half = synth.forest_cloud(200_000, seed=2, variant="J", return_half=True)
    ix.build(pts)
    lo, hi = pts.min(0), pts.max(0)
    rng = np.random.default_rng(3)
    # corner to corner and far away: the frontier fills up and falls back to depth-first steps
    a = np.concatenate([np.array([lo, [lo[0], hi[1], lo[2]]], np.float32), rng.uniform(lo, hi, (40, 3))]).astype(np.float32)
    b = np.concatenate([np.array([hi, [hi[0], lo[1], hi[2]]], np.float32), rng.uniform(lo, hi, (40, 3))]).astype(np.float32)
    _check_all(ix, pts, a, b, (0.0, 0.5), "crossing")
    fa = np.array([[1e6, 0, 0], [0, 1e6, 3], [1e6, 1e6, 1e6], [-1e6, 5, 1]], np.float32)
    fb = np.array([[-1e6, 0, 1], [0, 1e6 + 40, 3], [1e6, 1e6, 1e6], [1e6, -5, 2]], np.float32)
    _check_all(ix, pts, fa, fb, (0.5, 1e6), "far")
    shifted = (pts.astype(np.float64) + 1e6).astype(np.float32)
    ix.build(shifted)
    _check_all(ix, shifted, (a.astype(np.float64) + 1e6).astype(np.float32), (b.astype(np.float64) + 1e6).astype(np.float32),
               (0.5,), "shifted to 1e6")
    # non-finite endpoints and an empty index
    q = rng.uniform(-5, 5, (5000, 3)).astype(np.float32)
    a = rng.uniform(-5, 5, (12, 3)).astype(np.float32)
    b = rng.uniform(-5, 5, (12, 3)).astype(np.float32)
    bad = [np.nan, np.inf, -np.inf]
    for j in range(9):
        (a if j % 2 == 0 else b)[j, j % 3] = bad[j % 3]
    for cloud in (q, q[:0]):
        ix.build(cloud)
        for flags in FLAGS:
            for space in SPACES:
                gi, gt = _sweep(ix, a, b, 1.0, flags, space)
                assert (gi[:9] == -1).all() and np.isnan(gt[:9]).all(), (flags, space, gi, gt)
                if len(cloud) == 0:
                    assert (gi[9:] == -1).all() and np.isinf(gt[9:]).all()
        if len(cloud):
            _assert_same(*_sweep(ix, a, b, 1.0), *brute_sweep(cloud, a, b, 1.0), "finite rows")
    ix.build(q)
    for m in (0, 1):
        for space in SPACES:
            gi, gt = _sweep(ix, a[9:9 + m], b[9:9 + m], 1.0, PC_QUERY_AUTO, space)
            assert len(gi) == m and len(gt) == m
            if m:
                _assert_same(gi, gt, *brute_sweep(q, a[9:10], b[9:10], 1.0), "m = 1")


def _raw(ix, pa, pb, m, stride, space, flags=PC_QUERY_AUTO, r=0.5):
    """pc_sphere_sweep_batch on raw addresses (host numpy / device torch), returns (rc, idx, t)."""
    if space == PC_DEVICE:
        import torch
        oi = torch.empty(max(m, 1), dtype=torch.int32, device="cuda")
        ot = torch.empty(max(m, 1), dtype=torch.float32, device="cuda")
        rc = ix._L.pc_sphere_sweep_batch(ix._h, C.c_void_p(pa), C.c_void_p(pb), m, stride, space, flags, r,
                                         C.c_void_p(oi.data_ptr()), C.c_void_p(ot.data_ptr()))
        torch.cuda.synchronize()
        ix.sync()
        return rc, oi.cpu().numpy()[:m], ot.cpu().numpy()[:m]
    oi = np.empty(max(m, 1), np.int32)
    ot = np.empty(max(m, 1), np.float32)
    rc = ix._L.pc_sphere_sweep_batch(ix._h, C.c_void_p(pa), C.c_void_p(pb), m, stride, space, flags, r,
                                     C.c_void_p(oi.ctypes.data), C.c_void_p(ot.ctypes.data))
    return rc, oi[:m], ot[:m]


def test_sweep_stride_and_polyline(ix):
    import torch
    pts, half = synth.forest_cloud(200_000, seed=7, variant="L", return_half=True)
    ix.build(pts)
    rng = np.random.default_rng(8)
    # a random-walk polyline of 3001 points through the map: 3000 segments, b = a + stride (the rows overlap)
    steps = rng.normal(0, 0.4, (3001, 3)).astype(np.float32)
    poly = (np.cumsum(steps, 0) * np.float32(0.3) + np.array([0, 0, 1.5], np.float32)).astype(np.float32)
    ref = {r: brute_sweep(pts, poly[:-1], poly[1:], r) for r in (0.1, 0.5)}
    for stride in (3, 4):
        arr = np.zeros((len(poly), stride), np.float32)
        arr[:, :3] = poly
        if stride == 4:
            arr[:, 3] = np.nan                                       # the pad word is never read
        dev = torch.from_numpy(arr).cuda()
        for space in SPACES:
            base = arr.ctypes.data if space == PC_HOST else dev.data_ptr()
            for flags in FLAGS:
                for r, (ei, et) in ref.items():
                    rc, gi, gt = _raw(ix, base, base + 4 * stride, len(poly) - 1, stride, space, flags, r)
                    assert rc == L.PC_OK
                    _assert_same(gi, gt, ei, et, f"polyline stride={stride} space={space} flags={flags} r={r}")
        a4, b4 = arr[:-1].copy(), arr[1:].copy()
        for space in SPACES:
            _assert_same(*_sweep(ix, a4, b4, 0.5, PC_QUERY_SORTED, space), *ref[0.5], f"stride={stride} arrays space={space}")


def test_sweep_multi_chunk_host():
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
    bi, bt = brute_sweep(pts, a, b, 0.3)
    for flags in FLAGS:
        _assert_same(*h.sphere_sweep(a, b, 0.3, flags), bi, bt, f"multi-chunk flags={flags}")
    rc, gi, gt = _raw(h, starts.ctypes.data, starts.ctypes.data + 12, len(starts) - 1, 3, PC_HOST, r=0.3)
    assert rc == L.PC_OK
    _assert_same(gi, gt, *brute_sweep(pts, starts[:-1], starts[1:], 0.3), "multi-chunk polyline")
    h.close()


def test_sweep_1m_batch(ix):
    pts, half = synth.forest_cloud(200_000, seed=12, variant="J", return_half=True)
    ix.build(pts)
    rng = np.random.default_rng(13)
    m = 1_000_000
    starts = synth.rrt_queries(m, half, seed=14)
    a, b = _random_segments(rng, starts, rng.choice([0.0, 0.1, 1.0, 10.0], m))
    rows = rng.choice(m, 3000, replace=False)
    for r in (0.1, 0.5):
        bi, bt = brute_sweep(pts, a[rows], b[rows], r)
        ref = None
        for flags in FLAGS:
            for space in SPACES:
                gi, gt = _sweep(ix, a, b, r, flags, space)
                _assert_same(gi[rows], gt[rows], bi, bt, f"1M r={r} flags={flags} space={space}")
                if ref is None:
                    ref = (gi, gt)
                assert (gi == ref[0]).all() and (gt.view(np.uint32) == ref[1].view(np.uint32)).all(), \
                    f"1M r={r}: flags={flags} space={space} differ from the first path"


def test_sweep_relations(ix):
    pts, half = synth.forest_cloud(200_000, seed=11, variant="J", return_half=True)
    ix.build(pts)
    rng = np.random.default_rng(15)
    m = 40_000
    starts = synth.rrt_queries(m, half, seed=15)
    a, b = _random_segments(rng, starts, rng.choice([0.0, 0.2, 1.0, 5.0, 15.0], m))
    prev = None
    for r in (0.0, 0.05, 0.3, 0.5, 0.5000001, 1.0, 2.0):
        for flags in FLAGS:
            for space in SPACES:
                gi, gt = _sweep(ix, a, b, r, flags, space)
                # 1: t = 0 exactly when the range list of a is non-empty, and idx is its first entry
                off, hits = ix.range(a, r)
                inside = np.diff(off) > 0
                assert ((gt == 0) == inside).all(), f"t = 0 != range(a) non-empty (r={r})"
                assert (gi[inside] == hits[off[:-1][inside]]).all(), f"t = 0 idx != first range entry (r={r})"
                # 3: a non-empty range list at b means contact
                offb, _ = ix.range(b, r)
                assert (gi[np.diff(offb) > 0] >= 0).all(), f"range(b) non-empty without contact (r={r})"
                # 2: a == b gives the range answer at a, or no contact
                gi2, gt2 = _sweep(ix, a, a, r, flags, space)
                assert (gi2[inside] == hits[off[:-1][inside]]).all() and (gt2[inside] == 0).all()
                assert (gi2[~inside] == -1).all() and np.isinf(gt2[~inside]).all()
        # 4: monotone in the radius, bit for bit on the float output
        if prev is not None:
            assert (gt <= prev[1]).all(), f"t grew with the radius (r={r})"
            assert ((prev[0] < 0) | (gi >= 0)).all(), f"contact lost with a larger radius (r={r})"
        prev = (gi, gt)
    # the yes/no answer of pc_segment_nearest_batch(max_range = r) agrees outside a band of relative 2^-30 around R2
    rows = rng.choice(m, 4000, replace=False)
    _, sd = brute_segment(pts, a[rows], b[rows])
    for r in (0.05, 0.5, 2.0):
        gi, _ = _sweep(ix, a, b, r)
        si, _ = ix.segment_nearest(a, b, r)
        r2 = r * r
        clear = np.abs(sd - r2) > r2 * 2.0 ** -30
        assert clear.sum() > 0.99 * len(rows)
        assert ((gi[rows] >= 0) == (sd <= r2))[clear].all(), f"sweep contact != segment within r (r={r})"
        assert ((gi[rows] >= 0) == (si[rows] >= 0))[clear].all()


def test_sweep_refusals(ix):
    ix.build(np.zeros((10, 3), np.float32))
    a = np.zeros((4, 3), np.float32)
    pa = a.ctypes.data
    f = ix._L.pc_sphere_sweep_batch
    out_i = np.empty(4, np.int32)
    pi = C.c_void_p(out_i.ctypes.data)
    cases = [
        (pa, pa, 4, 5, PC_HOST, 0, 0.5),           # bad stride
        (None, pa, 4, 3, PC_HOST, 0, 0.5),         # NULL a
        (pa, None, 4, 3, PC_HOST, 0, 0.5),         # NULL b
        (pa, pa, 4, 3, L.PC_HOST_ASYNC, 0, 0.5),
        (pa, pa, 4, 3, L.PC_DEVICE_ASYNC, 0, 0.5),
        (pa, pa, 4, 3, PC_HOST, 1, 0.5),           # unknown flags
        (pa, pa, 4, 3, PC_HOST, 8, 0.5),
        (pa, pa, 4, 3, PC_HOST, 0, float("nan")),  # bad radius
        (pa, pa, 4, 3, PC_HOST, 0, -0.5),
        (pa, pa, 4, 3, PC_HOST, 0, float("inf")),
    ]
    for c in cases:
        rc = f(ix._h, C.c_void_p(c[0]) if c[0] else None, C.c_void_p(c[1]) if c[1] else None, c[2], c[3], c[4], c[5], c[6], pi, None)
        assert rc == L.PC_EINVAL, c
        assert b"pc_sphere_sweep_batch" in ix._L.pc_last_error(ix._h), c
    assert f(ix._h, None, None, 0, 3, PC_HOST, 0, 0.5, None, None) == L.PC_OK          # m = 0, NULL arrays
    with pytest.raises(PcError):
        ix.sphere_sweep(a, a, -1.0)
    ix.batch_shard(0, 2)
    try:
        assert f(ix._h, C.c_void_p(pa), C.c_void_p(pa), 4, 3, PC_HOST, 0, 0.5, pi, None) == L.PC_EINVAL
        assert b"pc_sphere_sweep_batch" in ix._L.pc_last_error(ix._h)
        with pytest.raises(PcError):
            ix.sphere_sweep(a, a, 0.5)
    finally:
        ix.batch_shard(0, 1)
