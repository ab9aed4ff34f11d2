"""GPU tests of pc_range_sorted_batch: offsets, indices and float32(d2) bit-equal with the fp64 brute force
(tests/range_sorted_brute.c) in both memory spaces, every list size class (sorted by the capturing warp, by a
CTA in shared memory, by a CTA in global memory), ties, tree shapes, degenerate inputs, capacity and refusals, plus the
relations to pc_range_batch (max_nn = 0) and pc_knn_batch (max_nn <= 32)."""
import ctypes as C

import numpy as np
import pytest

from range_sorted_brute import brute_range_sorted
from pointcloudtraj_b200 import PC_DEVICE, PC_HOST, PcError, PointCloudIndex, synth
from pointcloudtraj_b200 import _lib as L

pytestmark = pytest.mark.gpu

MAX_NN = (0, 1, 7, 32, 33, 100, 1000)


@pytest.fixture(scope="module")
def ix():
    h = PointCloudIndex(max_points=1 << 18, device=0)
    yield h
    h.close()


def _sorted(ix, q, r, max_nn=0, space=PC_HOST, cap=None):
    if space == PC_DEVICE:
        import torch
        tq = torch.from_numpy(np.ascontiguousarray(q)).cuda()
        off, idx, d2 = ix.range_sorted(tq, torch.as_tensor(np.atleast_1d(r), dtype=torch.float64).cuda(), max_nn, cap)
        return off.cpu().numpy(), idx.cpu().numpy(), d2.cpu().numpy()
    return ix.range_sorted(q, r, max_nn, cap)


def _truncate(off, idx, d2, max_nn):
    """the rows of a max_nn = 0 answer cut to max_nn"""
    if max_nn == 0:
        return off, idx, d2
    n = np.minimum(np.diff(off), max_nn)
    keep = np.concatenate([np.arange(off[j], off[j] + n[j]) for j in range(len(n))] + [np.zeros(0, np.int64)])
    o = np.zeros(len(off), np.int64)
    o[1:] = np.cumsum(n)
    return o, idx[keep], d2[keep]


def _assert_same(g, b, what=""):
    goff, gi, gd = g
    boff, bi, bd = b
    assert (goff == boff).all(), f"{what}: offsets differ at rows {np.nonzero(goff != boff)[0][:5]}"
    bad = np.nonzero((gi != bi) | (gd != bd.astype(np.float32)))[0]
    if len(bad):
        row = np.searchsorted(boff, bad[0], side="right") - 1
        raise AssertionError(f"{what}: {len(bad)} entries differ, first in row {row}: gpu {gi[boff[row]:boff[row + 1]][:12]} "
                             f"brute {bi[boff[row]:boff[row + 1]][:12]}")


def _forest_queries(pts, half, seed):
    rng = np.random.default_rng(seed)
    inside = synth.rrt_queries(400, half, seed=seed, lattice_frac=0.5)
    near = pts[rng.integers(0, len(pts), 400)] + rng.normal(0, 0.05, (400, 3)).astype(np.float32)
    far = synth.rrt_queries(100, half, seed=seed + 1) + np.float32(3 * half)
    return np.ascontiguousarray(np.concatenate([inside, near, far]).astype(np.float32))


@pytest.mark.parametrize("variant", ["J", "L"])
def test_range_sorted_forest_200k(ix, variant):
    pts, half = synth.forest_cloud(200_000, seed=11, variant=variant, return_half=True)
    q = _forest_queries(pts, half, 3)
    ix.build(pts)
    per_query = np.random.default_rng(2).uniform(0.0, 1.5, len(q))
    for r in (0.8, per_query):
        full = brute_range_sorted(pts, q, r)
        for max_nn in MAX_NN:
            b = _truncate(*full, max_nn)
            for space in (PC_HOST, PC_DEVICE):
                _assert_same(_sorted(ix, q, r, max_nn, space), b, f"{variant} scalar={np.ndim(r) == 0} max_nn={max_nn} space={space}")


def test_range_sorted_matches_range_and_knn(ix):
    pts, half = synth.forest_cloud(100_000, seed=8, variant="L", return_half=True)
    q = synth.rrt_queries(3000, half, seed=4, lattice_frac=0.5)
    ix.build(pts)
    for r in (0.35, np.random.default_rng(1).uniform(0.0, 0.7, len(q))):
        roff, ridx = ix.range(q, r)
        off, idx, d2 = ix.range_sorted(q, r)
        assert (off == roff).all()
        for j in range(len(q)):
            assert (np.sort(idx[off[j]:off[j + 1]]) == ridx[off[j]:off[j + 1]]).all(), j
    r = 0.35
    for k in (1, 3, 16, 32):
        ki, kd = ix.knn(q, k, r)
        off, idx, d2 = ix.range_sorted(q, r, k)
        n = np.diff(off)
        assert (n == (ki >= 0).sum(1)).all()
        mask = np.arange(k)[None, :] < n[:, None]
        assert (ki[mask] == idx).all() and (kd[mask] == d2).all(), k


def _radius_for_count(pts, c, want):
    """a radius whose inclusive ball around c holds exactly `want` points (distinct distances around the want-th)"""
    s = np.sort(((pts.astype(np.float64) - c.astype(np.float64)) ** 2).sum(1))
    assert s[want - 1] < s[want]
    r = np.sqrt(s[want - 1])
    while r * r < s[want - 1]:
        r = np.nextafter(r, np.inf)
    return r


def test_range_sorted_long_lists(ix):
    """Every size class of the sort: up to 512 hits (the capturing warp; one list of exactly 512 and one of 513), up to
    16384 (one CTA in shared memory) and beyond (one CTA in global memory), untruncated and cut to 50."""
    pts, half = synth.forest_cloud(150_000, seed=6, variant="J", return_half=True)
    ix.build(pts)
    q = synth.rrt_queries(24, half, seed=5)
    radii = np.array([0.5, 2.0, 4.0, 6.0, 9.0, 12.0, 40.0, 5.0] * 3)
    radii[1] = _radius_for_count(pts, q[1], 512)
    radii[9] = _radius_for_count(pts, q[9], 513)
    full = brute_range_sorted(pts, q, radii)
    sizes = np.diff(full[0])
    assert sizes[1] == 512 and sizes[9] == 513
    assert (sizes > 32768).any() and ((sizes > 513) & (sizes <= 16384)).any() and ((sizes > 0) & (sizes < 512)).any()
    for max_nn in (0, 50):
        b = _truncate(*full, max_nn)
        for space in (PC_HOST, PC_DEVICE):
            _assert_same(_sorted(ix, q, radii, max_nn, space), b, f"max_nn={max_nn} space={space}")


def test_range_sorted_ties(ix):
    # 100 coincident points: indices 0..99 at equal d2
    pts = np.tile(np.array([[1.0, 2.0, 3.0]], np.float32), (100, 1))
    q = np.array([[1.0, 2.0, 3.0], [0.0, 0.0, 0.0], [5.0, -1.0, 2.5]], np.float32)
    ix.build(pts)
    for space in (PC_HOST, PC_DEVICE):
        off, idx, d2 = _sorted(ix, q, 10.0, 0, space)
        assert off.tolist() == [0, 100, 200, 300] and (idx.reshape(3, 100) == np.arange(100)).all()
        assert (d2.reshape(3, 100) == d2.reshape(3, 100)[:, :1]).all()
        off, idx, d2 = _sorted(ix, q, 10.0, 7, space)
        assert (idx.reshape(3, 7) == np.arange(7)).all()
    # every point twice: d2 = 0 twice for a query on a point, the lower copy first
    rng = np.random.default_rng(7)
    base = rng.uniform(-1, 1, (500, 3)).astype(np.float32)
    pts = np.concatenate([base, base])
    q = np.concatenate([base[:100], rng.uniform(-1, 1, (100, 3)).astype(np.float32)])
    ix.build(pts)
    full = brute_range_sorted(pts, q, 0.4)
    for space in (PC_HOST, PC_DEVICE):
        g = _sorted(ix, q, 0.4, 0, space)
        _assert_same(g, full, f"duplicates space={space}")
        off, idx, d2 = g
        assert (idx[off[:100]] == np.arange(100)).all() and (idx[off[:100] + 1] == np.arange(500, 600)).all()
        assert (d2[off[:100]] == 0).all() and (d2[off[:100] + 1] == 0).all()


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 9, 33, 65, 4097])
def test_range_sorted_tree_shapes(ix, n):
    rng = np.random.default_rng(n)
    pts = rng.uniform(-2, 2, (n, 3)).astype(np.float32)
    q = np.concatenate([rng.uniform(-3, 3, (200, 3)), pts[: min(n, 50)]]).astype(np.float32)
    ix.build(pts)
    for r in (1.0, 10.0):
        full = brute_range_sorted(pts, q, r)
        for max_nn in (0, 5):
            for space in (PC_HOST, PC_DEVICE):
                _assert_same(_sorted(ix, q, r, max_nn, space), _truncate(*full, max_nn), f"n={n} r={r} max_nn={max_nn} space={space}")


def test_range_sorted_degenerate(ix):
    rng = np.random.default_rng(3)
    pts = rng.uniform(-1, 1, (2000, 3)).astype(np.float32)
    ix.build(pts)
    for space in (PC_HOST, PC_DEVICE):
        # empty batch
        off, idx, d2 = _sorted(ix, np.zeros((0, 3), np.float32), 1.0, 0, space)
        assert off.tolist() == [0] and len(idx) == 0 and len(d2) == 0
        # NaN range: an empty row; r = 0 with queries on points: the point itself (and nothing else)
        q = np.concatenate([pts[:50], rng.uniform(-1, 1, (50, 3)).astype(np.float32)])
        r = np.full(len(q), 0.3)
        r[::3] = np.nan
        r[1::3] = 0.0
        full = brute_range_sorted(pts, q, r)
        g = _sorted(ix, q, r, 0, space)
        _assert_same(g, full, f"nan / zero radii space={space}")
        assert (np.diff(g[0])[::3] == 0).all()
        on = [j for j in range(1, 50, 3)]
        assert (np.diff(g[0])[on] == 1).all() and (g[1][g[0][on]] == on).all()
        _assert_same(_sorted(ix, q, float("nan"), 0, space), (np.zeros(len(q) + 1, np.int64), np.zeros(0, np.int64), np.zeros(0)), "nan")
    # q_stride 4 (pcl::PointXYZ layout)
    q = rng.uniform(-1, 1, (300, 3)).astype(np.float32)
    q4 = np.concatenate([q, np.full((len(q), 1), 77.0, np.float32)], 1)
    full = brute_range_sorted(pts, q, 0.25)
    for max_nn in (0, 9):
        _assert_same(ix.range_sorted(q4, 0.25, max_nn), _truncate(*full, max_nn), f"stride 4 max_nn={max_nn}")
    # empty index
    ix.build(np.zeros((0, 3), np.float32))
    for space in (PC_HOST, PC_DEVICE):
        off, idx, d2 = _sorted(ix, q, 1.0, 0, space)
        assert (off == 0).all() and len(idx) == 0


def test_range_sorted_capacity(ix):
    pts, half = synth.forest_cloud(50_000, seed=3, variant="J", return_half=True)
    q = synth.rrt_queries(2000, half, seed=2)
    ix.build(pts)
    lib = L.load()
    rr = np.array([0.6])
    for max_nn in (0, 20):
        full = brute_range_sorted(pts, q, 0.6, max_nn)
        total = int(full[0][-1])
        assert total > 100
        # offsets only
        off = np.zeros(len(q) + 1, np.int64)
        rc = lib.pc_range_sorted_batch(ix._h, C.c_void_p(q.ctypes.data), len(q), 3, L.PC_HOST, C.c_void_p(rr.ctypes.data), 1, max_nn,
                                       C.c_void_p(off.ctypes.data), None, None, 0)
        assert rc == L.PC_OK and (off == full[0]).all()
        # too small a cap: PC_ECAP, offsets complete
        off[:] = -1
        oi = np.empty(total - 1, np.int32)
        od = np.empty(total - 1, np.float32)
        rc = lib.pc_range_sorted_batch(ix._h, C.c_void_p(q.ctypes.data), len(q), 3, L.PC_HOST, C.c_void_p(rr.ctypes.data), 1, max_nn,
                                       C.c_void_p(off.ctypes.data), C.c_void_p(oi.ctypes.data), C.c_void_p(od.ctypes.data), total - 1)
        assert rc == L.PC_ECAP and (off == full[0]).all()
        with pytest.raises(PcError):
            ix.range_sorted(q, 0.6, max_nn, cap=total - 1)
        # exactly enough, without d2
        oi = np.empty(total, np.int32)
        rc = lib.pc_range_sorted_batch(ix._h, C.c_void_p(q.ctypes.data), len(q), 3, L.PC_HOST, C.c_void_p(rr.ctypes.data), 1, max_nn,
                                       C.c_void_p(off.ctypes.data), C.c_void_p(oi.ctypes.data), None, total)
        assert rc == L.PC_OK and (off == full[0]).all() and (oi == full[1]).all()


def test_range_sorted_refusals(ix):
    ix.build(synth.uniform_cloud(1000))
    lib = L.load()
    q = np.zeros((4, 3), np.float32)
    rr = np.array([1.0])
    off = np.zeros(5, np.int64)
    oi = np.empty(64, np.int32)
    od = np.empty(64, np.float32)
    vp = lambda a: C.c_void_p(a.ctypes.data)
    for space, max_nn, pi, cap in ((L.PC_HOST_ASYNC, 0, vp(oi), 64), (L.PC_DEVICE_ASYNC, 0, vp(oi), 64), (7, 0, vp(oi), 64),
                                   (L.PC_HOST, -1, vp(oi), 64), (L.PC_HOST, 0, None, 64), (L.PC_HOST, 0, vp(oi), -1)):
        rc = lib.pc_range_sorted_batch(ix._h, vp(q), 4, 3, space, vp(rr), 1, max_nn, vp(off), pi, vp(od), cap)
        assert rc == L.PC_EINVAL, (space, max_nn, cap)
    with pytest.raises(PcError) as e:
        ix.range_sorted(q, 1.0, -1)
    assert e.value.code == L.PC_EINVAL
    # a pc_batch_shard handle answers every query, as pc_range_batch does
    pts = synth.uniform_cloud(1000)
    with PointCloudIndex(max_points=1000, device=0) as h:
        h.build(pts)
        h.batch_shard(0, 2)
        qq = synth.uniform_cloud(64)
        _assert_same(h.range_sorted(qq, 0.3), brute_range_sorted(pts, qq, 0.3), "shard handle")


def test_range_sorted_scale_1m_queries():
    pts, half = synth.forest_cloud(1_000_000, variant="J", return_half=True)
    q = synth.rrt_queries(1_000_000, half, seed=1)
    with PointCloudIndex(max_points=len(pts), device=0) as h:
        h.build(pts)
        off, idx, d2 = h.range_sorted(q, 0.5)
        roff, _ = h.range(q, 0.5)
        assert (off == roff).all()
        sub = np.sort(np.random.default_rng(0).choice(len(q), 2000, replace=False))
        boff, bi, bd = brute_range_sorted(pts, q[sub], 0.5)
        assert (np.diff(off)[sub] == np.diff(boff)).all()
        keep = np.concatenate([np.arange(off[j], off[j + 1]) for j in sub])
        assert (idx[keep] == bi).all() and (d2[keep] == bd.astype(np.float32)).all()
