"""GPU tests of pc_distance_field: the field is exactly what the composition it replaces returns -- the voxel centres made with
the contract's formula in numpy, pc_knn_batch(k = 1, max_range) (pc_nearest_batch when unbounded) on them, and the square root
of the fp64 d2 recomputed here from the winning point -- on the golden clouds and a 1 M-point forest, at every lattice shape
the brick tiling treats differently, inside, across and outside the cloud's box, at every kind of bound, with exact ties, on
degenerate clouds, in both memory spaces and across PC_HOST chunks; plus the brute force (tests/knn_brute.c) and a kd-tree
as independent oracles, nullable outputs, determinism, one launch per PC_DEVICE call and every refusal."""
import ctypes as C
import os

import numpy as np
import pytest

from knn_brute import brute_knn
from pointcloudtraj_b200 import PC_DEVICE, PC_HOST, PcError, PcLattice, PointCloudIndex, synth
from pointcloudtraj_b200 import _lib as L

pytestmark = pytest.mark.gpu

SHAPES = [(1, 1, 1), (5, 3, 7), (33, 1, 1), (1, 1, 65), (17, 9, 4)]
RANGES = [None, 0.0, 0.05, 0.5, 2.0, np.inf]


@pytest.fixture(scope="module")
def ix():
    h = PointCloudIndex(max_points=1 << 20, device=0)
    yield h
    h.close()


def centres(origin, voxel, dims):
    """The contract's float32 centres in output order (x fastest): (nz * ny * nx, 3)."""
    ax = [np.float32(float(origin[a]) + (np.arange(int(dims[a]), dtype=np.float64) + 0.5) * float(voxel)) for a in range(3)]
    z, y, x = np.meshgrid(ax[2], ax[1], ax[0], indexing="ij")
    return np.ascontiguousarray(np.stack([x.ravel(), y.ravel(), z.ravel()], 1).astype(np.float32))


def exact_dist(pts, c, idx):
    """sqrt of the reference's fp64 d2 of cloud[idx] against the centres, rounded once to float32; +inf where idx is -1."""
    p = pts[np.maximum(idx, 0)].astype(np.float64)
    cc = c.astype(np.float64)
    d2 = (p[:, 0] - cc[:, 0]) ** 2
    d2 = d2 + (p[:, 1] - cc[:, 1]) ** 2
    d2 = d2 + (p[:, 2] - cc[:, 2]) ** 2
    return np.where(idx >= 0, np.sqrt(d2).astype(np.float32), np.float32(np.inf))


def field(ix, origin, voxel, dims, r, space=PC_HOST):
    if space == PC_DEVICE:
        d, i = ix.distance_field(origin, voxel, dims, r, on_device=True)
        return d.cpu().numpy(), i.cpu().numpy()
    return ix.distance_field(origin, voxel, dims, r)


def check(ix, pts, origin, voxel, dims, r, what="", spaces=(PC_HOST, PC_DEVICE)):
    """The field against the knn composition (and nearest() when unbounded), in each space; returns (dist, idx) flat."""
    c = centres(origin, voxel, dims)
    ki, _ = ix.knn(c, 1, r)
    ki = ki[:, 0]
    if r is None:
        ni, _ = ix.nearest(c)
        assert (ni == ki).all(), what
    want = exact_dist(pts, c, ki)
    out = None
    for space in spaces:
        d, i = field(ix, origin, voxel, dims, r, space)
        assert d.shape == i.shape == (dims[2], dims[1], dims[0]), what
        d, i = d.ravel(), i.ravel()
        bad = np.nonzero(i != ki)[0]
        assert len(bad) == 0, f"{what} space={space}: {len(bad)} indices differ, first {bad[:5]}: {i[bad[:5]]} vs {ki[bad[:5]]}"
        bad = np.nonzero(d.view(np.uint32) != want.view(np.uint32))[0]
        assert len(bad) == 0, f"{what} space={space}: {len(bad)} distances differ, first {bad[:5]}: {d[bad[:5]]} vs {want[bad[:5]]}"
        if out is not None:
            assert (out[0].view(np.uint32) == d.view(np.uint32)).all() and (out[1] == i).all(), what
        out = (d, i)
    return out


def box_lattice(pts, dims, pad=0.0):
    """A lattice of the given dims over the finite points' box (grown by pad on every side)."""
    f = pts[np.isfinite(pts).all(1)]
    lo, hi = f.min(0).astype(np.float64) - pad, f.max(0).astype(np.float64) + pad
    voxel = float(max((hi - lo) / np.asarray(dims, np.float64)))
    return tuple(lo), voxel


@pytest.mark.parametrize("name", ["forest_jitter", "forest_lattice", "uniform"])
def test_golden_clouds(ix, golden_dir, name):
    pts = np.load(os.path.join(golden_dir, f"{name}.npz"))["pts"].astype(np.float32)
    ix.build(pts)
    for dims in SHAPES:
        origin, voxel = box_lattice(pts, dims, pad=0.5)
        for r in RANGES:
            check(ix, pts, origin, voxel, dims, r, f"{name} {dims} r={r}")


def test_forest_1m(ix):
    pts, half = synth.forest_cloud(1_000_000, seed=4, variant="J", return_half=True)
    ix.build(pts)
    f = pts[np.isfinite(pts).all(1)]
    mid = 0.5 * (f.min(0).astype(np.float64) + f.max(0).astype(np.float64))
    dims = (256, 256, 64)
    origin = (mid[0] - 12.8, mid[1] - 12.8, mid[2] - 3.2)
    d, i = check(ix, pts, origin, 0.1, dims, 2.0, "forest 1M 256x256x64 r=2")
    assert (i >= 0).mean() > 0.5
    # the unbounded field on the same lattice, PC_DEVICE only, and the bound as a truncation of it
    du, iu = check(ix, pts, origin, 0.1, dims, None, "forest 1M 256x256x64 unbounded", spaces=(PC_DEVICE,))
    keep = i >= 0
    assert (iu[keep] == i[keep]).all() and (du[keep] == d[keep]).all() and (du[~keep] > 2.0).all()
    for dims in SHAPES:
        for r in (None, 0.5):
            check(ix, pts, (mid[0] - 1.0, mid[1] + 0.3, 0.2), 0.1, dims, r, f"forest 1M {dims} r={r}")


def test_outside_the_box(ix):
    pts = synth.uniform_cloud(20_000, half=4.0, seed=2)
    ix.build(pts)
    for origin in [(3.0, 3.0, 6.0), (-2.0, 3.5, -1.0), (40.0, -50.0, 70.0), (-1e4, 1e4, 5.0)]:
        for dims in [(17, 9, 4), (5, 3, 7)]:
            for r in RANGES:
                check(ix, pts, origin, 0.25, dims, r, f"origin {origin} {dims} r={r}")


def test_brute_and_kdtree_oracles(ix):
    pts, half = synth.forest_cloud(100_000, seed=9, variant="L", return_half=True)
    ix.build(pts)
    dims = (40, 24, 12)
    origin, voxel = box_lattice(pts, dims)
    c = centres(origin, voxel, dims)
    for r in (None, 0.3):
        d, i = field(ix, origin, voxel, dims, r)
        bi, bd = brute_knn(pts, c, 1, r)
        assert (i.ravel() == bi[:, 0]).all(), f"r={r}"
        want = np.where(bi[:, 0] >= 0, np.sqrt(bd[:, 0]).astype(np.float32), np.float32(np.inf))
        assert (d.ravel() == want).all(), f"r={r}"
    from scipy.spatial import cKDTree
    dd, _ = cKDTree(pts.astype(np.float64)).query(c.astype(np.float64))
    d, _ = field(ix, origin, voxel, dims, None)
    assert np.allclose(d.ravel(), dd, rtol=1e-6, atol=0.0)


def test_exact_ties_lowest_index(ix):
    # integer points, each one present three times in a shuffled order; half-integer centres are equidistant from the 8
    # corners of their unit cell, integer centres lie on 3 copies of a point: the lowest original index must win every tie
    g = np.stack(np.meshgrid(np.arange(6), np.arange(5), np.arange(4), indexing="ij"), -1).reshape(-1, 3)
    pts = np.concatenate([g, g, g]).astype(np.float32)
    pts = pts[np.random.default_rng(1).permutation(len(pts))]
    ix.build(pts)
    for origin in [(0.0, 0.0, 0.0), (-0.5, -0.5, -0.5), (-2.0, -3.0, -1.0)]:
        for r in RANGES:
            d, i = check(ix, pts, origin, 1.0, (9, 8, 7), r, f"ties origin {origin} r={r}")
            c = centres(origin, 1.0, (9, 8, 7))
            bi, _ = brute_knn(pts, c, 1, r)
            assert (i == bi[:, 0]).all()
    # every half-integer centre inside the grid: 8 tied corners x 3 copies
    d, i = field(ix, (0.0, 0.0, 0.0), 1.0, (5, 4, 3), None)
    assert (d == np.float32(np.sqrt(0.75))).all()


def test_degenerate_clouds(ix):
    dims, origin = (9, 5, 6), (-1.0, -1.0, -1.0)
    rng = np.random.default_rng(3)
    one = np.array([[0.3, 0.2, 0.1]], np.float32)
    dup = np.repeat(rng.uniform(-1, 1, (5, 3)).astype(np.float32), 4, axis=0)[rng.permutation(20)]
    nan = rng.uniform(-1, 1, (300, 3)).astype(np.float32)
    nan[::7, rng.integers(0, 3)] = np.nan
    nan[5] = np.inf
    all_nan = np.full((50, 3), np.nan, np.float32)
    for name, pts in [("one", one), ("dup", dup), ("nan", nan), ("all-nan", all_nan)]:
        ix.build(pts)
        for r in RANGES:
            check(ix, pts, origin, 0.3, dims, r, f"{name} r={r}")
    d, i = field(ix, origin, 0.3, dims, None)
    assert (i == -1).all() and np.isinf(d).all()
    ix.build(np.zeros((0, 3), np.float32))
    for r in RANGES:
        for space in (PC_HOST, PC_DEVICE):
            d, i = field(ix, origin, 0.3, dims, r, space)
            assert (i == -1).all() and (d == np.inf).all()


def test_host_chunks_match_device():
    # 1024-voxel chunks: 37 x 11 voxels a layer puts one brick layer (1628 voxels) in every chunk of the PC_HOST pipeline
    os.environ["PC_HOST_CHUNK_QUERIES"] = "1024"
    try:
        h = PointCloudIndex(max_points=1 << 18, device=0)
    finally:
        del os.environ["PC_HOST_CHUNK_QUERIES"]
    try:
        pts = synth.forest_cloud(200_000, seed=5, variant="J")
        h.build(pts)
        for dims in [(37, 11, 29), (64, 64, 16), (1, 1, 65)]:
            origin, voxel = box_lattice(pts, dims)
            for r in (None, 0.5):
                check(h, pts, origin, voxel, dims, r, f"chunked {dims} r={r}")
    finally:
        h.close()


def _raw(ix, lat, r, space, dist, idx):
    vp = lambda a: C.c_void_p(0) if a is None else C.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)
    return ix._L.pc_distance_field(ix._h, C.byref(lat) if lat is not None else None, float(r), space, vp(dist), vp(idx))


def test_nullable_outputs_determinism_launches(ix):
    import torch
    pts = synth.forest_cloud(50_000, seed=7, variant="J")
    ix.build(pts)
    dims = (23, 18, 13)
    origin, voxel = box_lattice(pts, dims)
    lat = PcLattice.make(origin, voxel, dims)
    n = int(np.prod(dims))
    d0, i0 = field(ix, origin, voxel, dims, 0.4)
    for _ in range(3):
        d, i = field(ix, origin, voxel, dims, 0.4)
        assert (d.view(np.uint32) == d0.view(np.uint32)).all() and (i == i0).all()
    # each output NULL in turn, in both spaces: the other one is unchanged
    dist, idx = np.full(n, -7, np.float32), np.full(n, -7, np.int32)
    assert _raw(ix, lat, 0.4, PC_HOST, dist, None) == L.PC_OK and (dist == d0.ravel()).all()
    assert _raw(ix, lat, 0.4, PC_HOST, None, idx) == L.PC_OK and (idx == i0.ravel()).all()
    td, ti = torch.full((n,), -7.0, device="cuda"), torch.full((n,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    assert _raw(ix, lat, 0.4, PC_DEVICE, td, None) == L.PC_OK
    ix.sync()
    assert (td.cpu().numpy() == d0.ravel()).all() and (ti.cpu().numpy() == -7).all()
    assert _raw(ix, lat, 0.4, PC_DEVICE, None, ti) == L.PC_OK
    ix.sync()
    assert (ti.cpu().numpy() == i0.ravel()).all()
    # one kernel launch per PC_DEVICE call, nothing else: no ordering pass
    ix.launches(reset=True)
    for r in (-1.0, 0.4):
        assert _raw(ix, lat, r, PC_DEVICE, td, ti) == L.PC_OK
        assert ix.launches(reset=True) == 1
    ix.sync()
    # an empty lattice writes nothing and launches nothing
    for dims0 in [(0, 5, 5), (5, 0, 5), (5, 5, 0)]:
        idx[:] = -7
        assert _raw(ix, PcLattice.make(origin, voxel, dims0), 0.4, PC_HOST, dist, idx) == L.PC_OK
        assert (idx == -7).all()
        assert _raw(ix, PcLattice.make(origin, voxel, dims0), 0.4, PC_DEVICE, td, ti) == L.PC_OK
    assert ix.launches(reset=True) == 0


def test_refusals(ix):
    pts = synth.forest_cloud(10_000, seed=7, variant="J")
    ix.build(pts)
    dist, idx = np.empty(64, np.float32), np.empty(64, np.int32)
    ok = PcLattice.make((0.0, 0.0, 0.0), 0.1, (4, 4, 4))
    assert _raw(ix, ok, -1.0, PC_HOST, dist, idx) == L.PC_OK
    bad = [
        ((np.nan, 0.0, 0.0), 0.1, (4, 4, 4)), ((0.0, np.inf, 0.0), 0.1, (4, 4, 4)), ((0.0, 0.0, -np.inf), 0.1, (4, 4, 4)),
        ((0.0, 0.0, 0.0), 0.0, (4, 4, 4)), ((0.0, 0.0, 0.0), -0.1, (4, 4, 4)), ((0.0, 0.0, 0.0), np.nan, (4, 4, 4)),
        ((0.0, 0.0, 0.0), np.inf, (4, 4, 4)),
        ((0.0, 0.0, 0.0), 0.1, (-1, 4, 4)), ((0.0, 0.0, 0.0), 0.1, (4, 4, -4)), ((0.0, 0.0, 0.0), 0.1, (-1, 0, 4)),
        ((0.0, 0.0, 0.0), 0.1, (1 << 14, 1 << 14, (1 << 12) + 1)), ((0.0, 0.0, 0.0), 0.1, (1 << 62, 1 << 62, 4)),
        ((3e38, 0.0, 0.0), 1e38, (4, 4, 4)), ((0.0, -3.5e38, 0.0), 1.0, (4, 4, 4)), ((0.0, 0.0, 0.0), 1e300, (1, 1, 1)),
    ]
    for origin, voxel, dims in bad:
        assert _raw(ix, PcLattice.make(origin, voxel, dims), -1.0, PC_HOST, dist, idx) == L.PC_EINVAL, (origin, voxel, dims)
    assert _raw(ix, PcLattice.make((0.0, 0.0, 0.0), 0.1, (1 << 14, 1 << 14, 1 << 12)), -1.0, PC_HOST, None, None) == L.PC_OK
    assert _raw(ix, None, -1.0, PC_HOST, dist, idx) == L.PC_EINVAL
    assert _raw(ix, ok, float("nan"), PC_HOST, dist, idx) == L.PC_EINVAL
    for space in (L.PC_HOST_ASYNC, L.PC_DEVICE_ASYNC, 7):
        assert _raw(ix, ok, -1.0, space, dist, idx) == L.PC_EINVAL
    with pytest.raises(PcError):
        ix.distance_field((0.0, 0.0, 0.0), -1.0, (4, 4, 4))
    ix.batch_shard(0, 2)
    try:
        assert _raw(ix, ok, -1.0, PC_HOST, dist, idx) == L.PC_EINVAL
    finally:
        ix.batch_shard(0, 1)
    assert _raw(ix, ok, -1.0, PC_HOST, dist, idx) == L.PC_OK
