"""GPU parity tests for pc_range_batch (kd_nearest_range3), pc_sphere_gather and pc_clearance_batch (checkSafeTrajectory).

The wrapper reaches pc_range_batch and pc_sphere_gather in host memory only; the *_call helpers below call the C ABI in
either space (PC_DEVICE: every array a CUDA tensor) with outputs pre-filled by a sentinel, so that an entry the call should
not write is seen."""
import ctypes as C

import numpy as np
import pytest

import oracle
from pointcloudtraj_b200 import PcError, PcRadiusParams, PointCloudIndex, synth
from pointcloudtraj_b200 import _lib as L

pytestmark = pytest.mark.gpu

SPACES = (L.PC_HOST, L.PC_DEVICE)
SENTINEL = -7
GUARD = 16                      # list buffers are this much longer than the cap passed: nothing may land there


@pytest.fixture(scope="module")
def ix():
    h = PointCloudIndex(max_points=1 << 18, device=0)
    yield h
    h.close()


@pytest.fixture(scope="module")
def forest():
    """The clearance tests' map and the CPU kd-tree over it."""
    pts, half = synth.forest_cloud(150_000, seed=6, variant="J", return_half=True)
    return pts, half, oracle.KdOracle().build(pts, np.random.default_rng(1).permutation(len(pts)))


def _vp(a):
    return C.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)


def _in_space(arrays, space):
    """The arrays as they are (PC_HOST) or as CUDA tensors (PC_DEVICE), copies finished."""
    if space == L.PC_HOST:
        return list(arrays)
    import torch
    out = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]
    torch.cuda.synchronize()
    return out


def _home(a):
    return a if isinstance(a, np.ndarray) else a.cpu().numpy()


def _brute_range(pts, q, r):
    """Exact fp64 sets {i : d2(i) <= r*r} in the reference's operation order, ascending index."""
    P = pts.astype(np.float64)
    out = []
    r = np.broadcast_to(np.asarray(r, np.float64), (len(q),))
    for k in range(len(q)):
        d = P - q[k].astype(np.float64)
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        out.append(np.nonzero(d2 <= r[k] * r[k])[0])
    return out


def _lists(off, idx):
    return [idx[off[k]:off[k + 1]] for k in range(len(off) - 1)]


def _csr(lists):
    off = np.zeros(len(lists) + 1, np.int64)
    off[1:] = np.cumsum([len(x) for x in lists])
    return off, np.concatenate(lists).astype(np.int32)


def _range_call(ix, q, r, space, cap, lists=True):
    """pc_range_batch in `space` (the range array too); lists=False passes out_idx = NULL.  -> (rc, offsets, idx[cap + GUARD])"""
    q = np.ascontiguousarray(q, np.float32)
    rr = np.ascontiguousarray(np.atleast_1d(r), np.float64)
    dq, dr, doff, didx = _in_space([q, rr, np.full(len(q) + 1, SENTINEL, np.int64), np.full(cap + GUARD, SENTINEL, np.int32)], space)
    rc = ix._L.pc_range_batch(ix._h, _vp(dq), len(q), q.shape[1], space, _vp(dr), int(rr.size == 1), _vp(doff),
                              _vp(didx) if lists else None, cap)
    ix.sync()
    return rc, _home(doff), _home(didx)


def _check_range(ix, pts, q, r, space, what):
    """The lists at cap == total equal the brute force, and nothing lands past the cap; the offsets-only call and
    cap == total - 1 (PC_ECAP) give the same complete offsets."""
    off, want = _csr(_brute_range(pts, q[:, :3], r))
    total = int(off[-1])
    rc, goff, gidx = _range_call(ix, q, r, space, total)
    assert rc == L.PC_OK, f"{what}: {ix._L.pc_last_error(ix._h).decode()}"
    assert (goff == off).all(), f"{what}: offsets differ at rows {np.nonzero(goff != off)[0][:5]}"
    bad = np.nonzero(gidx[:total] != want)[0]
    assert bad.size == 0, f"{what}: {bad.size} list entries differ, first in row {np.searchsorted(off, bad[:1], 'right') - 1}"
    assert (gidx[total:] == SENTINEL).all(), f"{what}: written past the cap"
    rc, goff, gidx = _range_call(ix, q, r, space, 0, lists=False)
    assert rc == L.PC_OK and (goff == off).all() and (gidx == SENTINEL).all(), f"{what}: offsets only"
    if total > 0:
        rc, goff, gidx = _range_call(ix, q, r, space, total - 1)
        assert rc == L.PC_ECAP and (goff == off).all() and (gidx[total - 1:] == SENTINEL).all(), f"{what}: cap = total - 1"


@pytest.mark.parametrize("name", ["forest_lattice", "forest_jitter", "uniform"])
def test_range_golden(ix, golden_dir, name):
    g = np.load(f"{golden_dir}/{name}.npz")
    pts, q, r = g["pts"], g["range_q"], float(g["range_r"])
    ix.build(pts)
    off, idx = ix.range(q, r)
    gpu = _lists(off, idx)
    ref = _lists(g["range_off"], g["range_idx"])
    brute = _brute_range(pts, q, r)
    for k in range(len(q)):
        assert (np.diff(gpu[k]) > 0).all()                        # ascending original index, no duplicates
        assert (gpu[k] == brute[k]).all() if len(gpu[k]) == len(brute[k]) else False
        # the reference may miss points at exactly `range` across a split plane (kdtree.c:283), never more
        assert np.isin(ref[k], gpu[k]).all()
    if name != "forest_lattice":
        assert (off == g["range_off"]).all()                      # tie-free inputs: identical sets
        assert all((np.sort(ref[k]) == gpu[k]).all() for k in range(len(q)))


def test_range_known_answers(ix):
    # SURVEY 8c-5: points (0.5,5,5), (0.5,0,0); the point at exactly range 1 is found from BOTH sides here
    ix.build(np.array([[0.5, 5, 5], [0.5, 0, 0]], np.float32))
    off, idx = ix.range(np.array([[-0.5, 0, 0], [1.5, 0, 0], [9, 9, 9]], np.float32), 1.0)
    assert off.tolist() == [0, 1, 2, 2] and idx.tolist() == [1, 1]
    # empty index, empty batch
    ix.build(np.zeros((0, 3), np.float32))
    off, idx = ix.range(np.zeros((3, 3), np.float32), 2.0)
    assert off.tolist() == [0, 0, 0, 0] and idx.size == 0
    off, idx = ix.range(np.zeros((0, 3), np.float32), 2.0)
    assert off.tolist() == [0]


def test_range_forest_vs_oracle_and_capacity(ix):
    pts, half = synth.forest_cloud(120_000, seed=6, variant="J", return_half=True)
    q = synth.rrt_queries(3000, half, seed=2)
    radii = np.random.default_rng(0).uniform(0.2, 3.0, len(q))          # planner uses 2 * radius <= 3 m
    ix.build(pts)
    off, idx = ix.range(q, radii)
    ko = oracle.KdOracle().build(pts, np.random.default_rng(1).permutation(len(pts)))
    roff, ridx = ko.range(q, radii)
    assert (off == roff).all()
    gl, rl = _lists(off, idx), _lists(roff, ridx)
    assert all((np.sort(rl[k]) == gl[k]).all() for k in range(len(q)))
    assert off[-1] > 100_000                                            # a real workload, not an empty check
    # duplicates of the last point pad the last leaf: they must not be reported twice
    last = pts[-1:]
    o2, i2 = ix.range(last, 1e-3)
    assert (np.diff(i2) > 0).all() and (len(pts) - 1) in i2
    # capacity overflow -> PC_ECAP, offsets still complete
    with pytest.raises(PcError) as e:
        ix.range(q, radii, cap=1000)
    assert e.value.code == -4


def test_range_long_lists(ix):
    """Lists beyond the in-warp sort (1024 hits) are sorted by one CTA each (up to 32768 hits), beyond that by the slow path:
    every size class gives the brute-force set in ascending order."""
    pts, half = synth.forest_cloud(150_000, seed=6, variant="J", return_half=True)
    ix.build(pts)
    q = synth.rrt_queries(24, half, seed=5)
    radii = np.array([0.5, 2.0, 4.0, 6.0, 9.0, 12.0, 40.0, 5.0] * 3)
    off, idx = ix.range(q, radii)
    brute = _brute_range(pts, q, radii)
    sizes = np.diff(off)
    assert (sizes > 32768).any() and ((sizes > 1024) & (sizes <= 32768)).any() and (sizes <= 1024).any()
    for k in range(len(q)):
        assert len(brute[k]) == sizes[k] and (idx[off[k]:off[k + 1]] == brute[k]).all()


# list lengths at the ends of each path of pc_range_batch: captured and sorted by the counting pass (<= PC_RCAP_HITS = 512),
# walked again and sorted by one CTA in shared memory (<= PC_RLONG_CAP = 32768), sorted by a single thread beyond
RANGE_CLASSES = (0, 1, 511, 512, 513, 32768, 32769, 70_000)


def test_range_list_classes_both_spaces(ix):
    """One query per length of RANGE_CLASSES, with exactly that many points within 1 mm of it (the 32768 of them coincident),
    queries 3 m apart and every other point at least 1.5 m away, the cloud shuffled so that each list is sorted for real.  Both
    spaces, a scalar range and per-query ranges, stride 3 and 4, and the capacity calls around the total."""
    rng = np.random.default_rng(17)
    q = np.zeros((len(RANGE_CLASSES), 3), np.float32)
    q[:, 0] = 3.0 * np.arange(len(q))
    q[:, 2] = 1.5
    parts = [np.tile(c, (n, 1)) if n == 32768 else c + rng.uniform(-5e-4, 5e-4, (n, 3)).astype(np.float32)
             for c, n in zip(q, RANGE_CLASSES)]
    parts.append(synth.uniform_cloud(20_000, half=30.0, seed=3, z=(3.0, 10.0)))
    pts = np.concatenate(parts)
    pts = np.ascontiguousarray(pts[rng.permutation(len(pts))])
    ix.build(pts)
    per_query = rng.uniform(2e-3, 1.0, len(q))
    for r in (0.5, per_query):
        assert [len(x) for x in _brute_range(pts, q, r)] == list(RANGE_CLASSES)
    q4 = np.concatenate([q, np.full((len(q), 1), 77.0, np.float32)], 1)
    for space in SPACES:
        _check_range(ix, pts, q, 0.5, space, f"scalar, space {space}")
        _check_range(ix, pts, q, per_query, space, f"per-query, space {space}")
        _check_range(ix, pts, q4, per_query, space, f"stride 4, space {space}")


def test_range_edge_rows_both_spaces(ix):
    """NaN and infinite query rows give empty rows and leave their neighbours alone; per-query ranges of 0 (a point and its
    coincident copies), -0.0, negative values (the set of |r|: the test is d2 <= r*r) and NaN (an empty row)."""
    rng = np.random.default_rng(23)
    pts = synth.uniform_cloud(30_000, half=4.0, seed=8, z=(0.0, 4.0))
    pts[100:110] = pts[7]
    ix.build(pts)
    q = synth.uniform_cloud(600, half=4.5, seed=9, z=(-0.5, 4.5))
    q[::7] = pts[rng.integers(len(pts), size=len(q[::7]))]
    q[0] = pts[7]
    special = [(np.nan, 0, 1), (np.inf, 0, 1), (0, -np.inf, 1), (1, 2, np.nan), (np.inf, np.inf, np.inf), (-np.inf, np.nan, 0)]
    rows = 5 + 13 * np.arange(len(special))
    q[rows] = special
    r = rng.uniform(0.05, 0.6, len(q))
    r[::5] = 0.0
    r[1::5] *= -1.0
    r[2::9] = np.nan
    r[3::11] = -0.0
    brute = _brute_range(pts, q, r)
    assert len(brute[0]) == 11 and all(len(brute[k]) == 0 for k in rows)
    assert sum(len(brute[k]) for k in range(1, len(q), 5)) > 0
    for space in SPACES:
        _check_range(ix, pts, q, r, space, f"per-query, space {space}")
        _check_range(ix, pts, q, -0.3, space, f"negative scalar, space {space}")
        _check_range(ix, pts, q, np.nan, space, f"NaN scalar, space {space}")


# ---- sensing gather --------------------------------------------------------------------------------------------------------
def _gather_call(ix, centre, radius, space, cap, lists=True):
    """pc_sphere_gather with out_idx in `space`; lists=False passes out_idx = NULL.  -> (rc, count, idx[cap + GUARD])"""
    c = (C.c_double * 3)(*[float(v) for v in centre])
    didx, = _in_space([np.full(cap + GUARD, SENTINEL, np.int32)], space)
    cnt = C.c_int64(SENTINEL)
    rc = ix._L.pc_sphere_gather(ix._h, c, float(radius), space, _vp(didx) if lists else None, cap, C.byref(cnt))
    ix.sync()
    return rc, cnt.value, _home(didx)


def _brute_gather(pts, centre, radius, f32_centre=True):
    """{i : d2(i) <= radius^2} from the centre cast to float32 (as the header promises) or from the double centre."""
    c = np.asarray(centre, np.float64)
    c = c.astype(np.float32).astype(np.float64) if f32_centre else c
    d2 = np.zeros(len(pts))
    for a in range(3):
        d = pts[:, a].astype(np.float64) - c[a]
        d2 = d2 + d * d
    return np.nonzero(d2 <= radius * radius)[0]


def _check_gather(ix, pts, centre, radius, space, what):
    """Count only, cap == count (the list equals the brute force, nothing lands past it) and cap == count - 1 (PC_ECAP with
    the count still right)."""
    want = _brute_gather(pts, centre, radius)
    n = len(want)
    rc, cnt, got = _gather_call(ix, centre, radius, space, 0, lists=False)
    assert rc == L.PC_OK and cnt == n, f"{what}: count only gave {rc}, {cnt} for {n}"
    rc, cnt, got = _gather_call(ix, centre, radius, space, n)
    assert rc == L.PC_OK and cnt == n, f"{what}: cap = count gave {rc}, {cnt} for {n}"
    bad = np.nonzero(got[:n] != want)[0]
    assert bad.size == 0 and (got[n:] == SENTINEL).all(), f"{what}: {bad.size} entries differ, first at {bad[:3]}"
    if n > 0:
        rc, cnt, got = _gather_call(ix, centre, radius, space, n - 1)
        assert rc == L.PC_ECAP and cnt == n and (got[n - 1:] == SENTINEL).all(), f"{what}: cap = count - 1"
    return want


def test_sphere_gather_spaces_capacity_and_edges(ix):
    """Both spaces, the count-only call and the capacity edges, on a map with non-finite points (never returned), coincident
    points (radius 0 returns them all; a negative radius is its absolute value) and points placed so that the float32 centre
    and the double centre the caller passes disagree: the search runs from the float32 one."""
    pts, half = synth.forest_cloud(60_000, seed=5, variant="J", return_half=True)
    centre = (0.1, 0.2, 0.3)                                  # no coordinate is a float32 number
    cf = np.array(centre, np.float32)
    assert (cf.astype(np.float64) > np.array(centre)).all()
    edge = cf.copy()
    edge[0] += np.float32(0.75)                               # farther from the double centre than from the float32 one
    r_edge = float(edge[0]) - float(cf[0])
    c0 = np.array([2.5, -1.25, 1.0], np.float32)
    extra = np.array([cf, edge] + [c0] * 6 + [(np.nan, 0, 1), (np.inf, 0, 1), (0, -np.inf, 1), (np.nan, np.nan, np.nan),
                                              (np.inf, -np.inf, np.inf)], np.float32)
    pts = np.concatenate([pts[:30_000], extra, pts[30_000:]])
    finite = np.isfinite(pts).all(1)
    ix.build(pts)
    for space in SPACES:
        got = _check_gather(ix, pts, centre, 0.0, space, f"radius 0 at the float32 centre, space {space}")
        assert got.tolist() == [30_000] and len(_brute_gather(pts, centre, 0.0, f32_centre=False)) == 0
        got = _check_gather(ix, pts, centre, r_edge, space, f"float32 centre, space {space}")
        assert 30_001 in got and 30_001 not in _brute_gather(pts, centre, r_edge, f32_centre=False)
        got = _check_gather(ix, pts, c0, 0.0, space, f"coincident points, space {space}")
        assert got.tolist() == list(range(30_002, 30_008))
        got = _check_gather(ix, pts, c0, -2.5, space, f"negative radius, space {space}")
        assert (got == _brute_gather(pts, c0, 2.5)).all() and len(got) > 100
        got = _check_gather(ix, pts, (0.0, 0.0, 2.0), 1e4, space, f"the whole map, space {space}")
        assert (got == np.nonzero(finite)[0]).all()
    with pytest.raises(PcError) as e:
        ix.sphere_gather(centre, float("nan"))
    assert e.value.code == L.PC_EINVAL


@pytest.mark.parametrize("n", [255, 256, 65535, 65536, (1 << 24) + 1])
def test_sphere_gather_key_widths(n):
    """The gather sorts its hits by original index on 8, 16, 24 or 32 key bits, chosen from the cloud size: each size here is
    the last or the first of a width.  The whole cloud (its highest index included) and a ball around the last point come
    back in ascending order, in both spaces."""
    pts = synth.uniform_cloud(n, half=16.0, seed=n % 1000)
    with PointCloudIndex(max_points=n, device=0) as h:
        h.build(pts)
        for space in SPACES:
            _check_gather(h, pts, (0.0, 0.0, 4.0), 1e3, space, f"n={n} whole cloud, space {space}")
            got = _check_gather(h, pts, pts[-1], 6.0, space, f"n={n} around the last point, space {space}")
            assert got[-1] == n - 1


# ---- clearance ---------------------------------------------------------------------------------------
def _clearance_oracle(ko, P, tr, t_now, horizon, dt=0.02):
    first, order, T, off, coef = tr["traj_first_seg"], tr["seg_order"], tr["seg_T"], tr["seg_coef_off"], tr["coef"]
    res = []
    for t in range(len(first) - 1):
        segs = range(first[t], first[t + 1])
        ld = 3 * (int(order[first[t]:first[t + 1]].max()) + 1) if len(segs) else 1
        mat = np.zeros((len(segs), ld))
        for r_, s in enumerate(segs):
            c = coef[off[s]:off[s + 1]]
            mat[r_, : len(c)] = c
        res.append(ko.check_safe_trajectory(P, order[first[t]:first[t + 1]], T[first[t]:first[t + 1]], mat,
                                            t_now=float(t_now[t]), stop_time=horizon, dt=dt, cap=8192))
    return res


CLR_START = (0.0, 0.0, 2.0)
CLR_P = PcRadiusParams.make(0.25, 1.5, 30.0, CLR_START)
CLR_OP = oracle.RadiusParams.make(0.25, 1.5, 30.0, CLR_START)


def _edge_t_now(tr):
    """Per trajectory, in turn: 0, negative, exactly the first segment's T (the skip test is a strict >), the sum of the first
    two T, one ulp past the first T (the walk starts ulps into the second segment), past the end, and a random time."""
    first, T = tr["traj_first_seg"], tr["seg_T"]
    n = len(first) - 1
    total = np.add.reduceat(T, first[:-1])
    t1 = T[first[:-1]]
    t2 = t1 + np.where(np.diff(first) > 1, T[np.minimum(first[:-1] + 1, len(T) - 1)], 0.0)
    cases = np.stack([np.zeros(n), np.full(n, -1.5), t1, t2, np.nextafter(t1, np.inf), total + 0.5,
                      np.random.default_rng(n).uniform(0, total)])
    return cases[np.arange(n) % len(cases), np.arange(n)]


def _prefix(tr, n):
    """The first n trajectories and only their segments and coefficients."""
    s = int(tr["traj_first_seg"][n])
    off = tr["seg_coef_off"][: s + 1]
    return dict(traj_first_seg=tr["traj_first_seg"][: n + 1], seg_order=tr["seg_order"][:s], seg_T=tr["seg_T"][:s],
                seg_coef_off=off, coef=tr["coef"][: off[-1]])


def _clearance_call(ix, tr, t_now, dt, horizon, space, n_samples=True):
    """pc_clearance_batch in `space` (the pc_traj records too); n_samples=False passes out_n_samples = NULL.
    -> (first_hit, min_radius, n_samples or None)"""
    first = tr["traj_first_seg"]
    n = len(first) - 1
    traj = np.zeros(n, dtype=[("first_seg", "<i4"), ("num_seg", "<i4"), ("t_now", "<f8")])
    traj["first_seg"], traj["num_seg"], traj["t_now"] = first[:-1], np.diff(first), t_now
    d = _in_space([traj.view(np.uint8), tr["seg_order"].astype(np.int32), tr["seg_T"], tr["seg_coef_off"], tr["coef"],
                   np.full(n, SENTINEL, np.int32), np.full(n, SENTINEL, np.float32), np.full(n, SENTINEL, np.int32)], space)
    rc = ix._L.pc_clearance_batch(ix._h, _vp(d[0]), n, _vp(d[1]), _vp(d[2]), _vp(d[3]), len(tr["seg_order"]), _vp(d[4]),
                                  len(tr["coef"]), space, float(dt), float(horizon), C.byref(CLR_P), _vp(d[5]), _vp(d[6]),
                                  _vp(d[7]) if n_samples else None)
    assert rc == L.PC_OK, ix._L.pc_last_error(ix._h).decode()
    ix.sync()
    fh, mr, ns = (_home(a) for a in d[5:])
    if not n_samples:
        assert (ns == SENTINEL).all()
    return fh, mr, ns if n_samples else None


def _assert_clearance(got, ref, what):
    """Exact: the kernel's powers are the correctly rounded u^j (double-double), like libm's pow in the oracle, so the float32
    sample positions, every radius and therefore the first colliding sample are identical (DESIGN.md "Clearance")."""
    fh, mr, ns = got
    r_ns = np.array([r["n_samples"] for r in ref])
    r_mr = np.array([r["min_radius"] for r in ref])
    if ns is not None:
        bad = np.nonzero(ns != r_ns)[0]
        assert bad.size == 0, f"{what}: sample counts differ at {bad[:5]}: {ns[bad[:5]]} vs {r_ns[bad[:5]]}"
    bad = np.nonzero(fh != np.array([r["first_hit"] for r in ref]))[0]
    assert bad.size == 0, f"{what}: first hits differ at {bad[:5]}"
    fin = np.isfinite(r_mr)                                         # trajectories without samples report +inf
    assert (np.isposinf(mr) == ~fin).all(), f"{what}: +inf rows differ"
    bad = np.nonzero(mr[fin] != r_mr[fin].astype(np.float32))[0]
    assert bad.size == 0, f"{what}: min radius differs at {np.nonzero(fin)[0][bad[:5]]}"


# the walk's edges: dt longer than any segment (3.5 s), an exact dt whose multiples reach the horizon exactly (the stop test is
# t_accu > horizon), and horizons of 0 and below (no sample); every case with the t_now edges of _edge_t_now and orders 1..12
@pytest.mark.parametrize("horizon,n_traj,dt", [(2.0, 300, 0.02), (20.0, 60, 0.02), (3.0, 140, 0.02), (2.0, 140, 0.125),
                                               (12.0, 140, 3.5), (0.0, 140, 0.02), (-1.0, 140, 0.02)],
                         ids=["2.0-300", "20.0-60", "3.0-140", "2.0-140-dt0.125", "12.0-140-dt3.5", "0.0-140", "-1.0-140"])
def test_clearance_vs_oracle(ix, forest, horizon, n_traj, dt):
    """Both spaces (PC_DEVICE also without n_samples), every Bezier order 1..12, against the CPU checkSafeTrajectory."""
    pts, half, ko = forest
    ix.build(pts)
    tr = synth.bezier_trajectories(n_traj, half * 0.9, seed=3, order_range=(1, 12))
    assert set(tr["seg_order"].tolist()) == set(range(1, 13))
    t_now = _edge_t_now(tr)
    ref = _clearance_oracle(ko, CLR_OP, tr, t_now, horizon, dt)
    r_ns = np.array([r["n_samples"] for r in ref])
    r_fh = np.array([r["first_hit"] for r in ref])
    if horizon > 0:
        assert r_ns.max() >= min(int(horizon / dt) - 1, 400) and (r_fh >= 0).any() and (r_fh < 0).any()
        assert (r_ns[5::7] == 0).all()                          # t_now past the end
    else:
        assert (r_ns == 0).all()
    for space, with_ns in ((L.PC_HOST, True), (L.PC_DEVICE, True), (L.PC_DEVICE, False)):
        _assert_clearance(_clearance_call(ix, tr, t_now, dt, horizon, space, with_ns), ref, f"space {space}, n_samples {with_ns}")


def test_clearance_kernel_by_schedule_size(ix, forest):
    """The flat path (3 launches) holds a schedule of horizon / dt + 4 samples per trajectory and gives way to the
    one-warp-per-trajectory kernel (1 launch) above 2^27 of them: at horizon 1000 s and dt 0.02, 2684 trajectories take the
    first and 2700 the second.  Both against the CPU checkSafeTrajectory, in both spaces."""
    pts, half, ko = forest
    ix.build(pts)
    tr = synth.bezier_trajectories(2700, half * 0.9, seed=14, seg_range=(1, 3), order_range=(1, 12), T_range=(0.2, 1.0))
    t_now = _edge_t_now(tr)
    ref = _clearance_oracle(ko, CLR_OP, tr, t_now, 1000.0, 0.02)
    for n, launches in ((2684, 3), (2700, 1)):
        for space in SPACES:
            n0 = ix.launches()
            got = _clearance_call(ix, _prefix(tr, n), t_now[:n], 0.02, 1000.0, space)
            assert ix.launches() - n0 == launches, (n, space)
            _assert_clearance(got, ref[:n], f"{n} trajectories, space {space}")


def _staged_bytes(n_traj, n_seg, n_coef):
    """What a PC_HOST pc_clearance_batch uploads, each array padded to 256 B: up to 256 KB it travels through one pinned
    staging block (clearance_host.inl), beyond that array by array."""
    pad = lambda b: -(-b // 256) * 256
    return pad(16 * n_traj) + pad(4 * n_seg) + 2 * pad(8 * n_seg) + pad(8 * n_coef)


def test_clearance_host_staging_threshold(ix, forest):
    pts, half, ko = forest
    ix.build(pts)
    tr = synth.bezier_trajectories(400, half * 0.9, seed=15, order_range=(1, 12))
    first, off = tr["traj_first_seg"], tr["seg_coef_off"]
    size = [_staged_bytes(n, int(first[n]), int(off[first[n]])) for n in range(len(first))]
    n = max(k for k in range(len(size)) if size[k] <= 1 << 18)
    assert n < 400 and size[n + 1] > 1 << 18
    t_now = _edge_t_now(tr)
    ref = _clearance_oracle(ko, CLR_OP, tr, t_now, 4.0, 0.02)
    for m in (n, n + 1):
        _assert_clearance(_clearance_call(ix, _prefix(tr, m), t_now[:m], 0.02, 4.0, L.PC_HOST), ref[:m], f"{m} trajectories")


def test_clearance_edge_cases(ix):
    pts = np.array([[5.0, 0, 1.0]], np.float32)
    ix.build(pts)
    P = PcRadiusParams.make(0.25, 1.5, 30.0, (0, 0, 1))
    T, n = 4.0, 4
    xs = np.linspace(0, 8, n + 1) / T
    coef = np.concatenate([xs, np.zeros(n + 1), np.full(n + 1, 1.0 / T)])
    first = np.array([0, 1, 1], np.int32)                          # second trajectory has no segments
    fh, mr, ns = ix.clearance(first, [n], [T], [0, len(coef)], coef, P, t_now=[0.0, 0.0], horizon=10.0)
    ko = oracle.KdOracle().build(pts)
    ref = ko.check_safe_trajectory(oracle.RadiusParams.make(0.25, 1.5, 30.0, (0, 0, 1)), [n], [T], coef[None, :], 0.0, 10.0)
    assert ns.tolist() == [ref["n_samples"], 0] == [200, 0]
    assert fh.tolist() == [ref["first_hit"], -1]
    assert mr[0] == np.float32(ref["min_radius"]) and np.isinf(mr[1])
    # empty cloud: every sample gets max_radius - search_margin (corridor_finder.cpp:118-120), no collision
    ix.build(np.zeros((0, 3), np.float32))
    fh, mr, ns = ix.clearance(first[:2], [n], [T], [0, len(coef)], coef, P, horizon=1.0)
    assert fh.tolist() == [-1] and mr.tolist() == [1.25]
    # bad arguments are rejected, not executed
    with pytest.raises(PcError):
        ix.clearance(first[:2], [13], [T], [0, len(coef)], coef, P)
    with pytest.raises(PcError):
        ix.clearance(first[:2], [n], [T], [0, len(coef)], coef, P, dt=0.0)


def test_sphere_gather_matches_brute_force(ix):
    """pc_sphere_gather: the LiDAR-mode observation (camera_sensor.cpp:133-145) = all points within max_dist of the sensor."""
    pts, half = synth.forest_cloud(250_000, seed=4, variant="J", return_half=True)
    ix.build(pts)
    for center, radius in (((1.0, -2.0, 2.0), 20.0), ((half, half, 0.0), 6.5), ((0.0, 0.0, 100.0), 5.0), ((0.0, 0.0, 2.0), 1e4)):
        got = ix.sphere_gather(center, radius)
        c = np.array(center, np.float32).astype(np.float64)
        d = pts.astype(np.float64) - c
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        want = np.nonzero(d2 <= radius * radius)[0]
        assert got.dtype == np.int32 and (got == want).all() if len(got) == len(want) else False
    ix.build(np.zeros((0, 3), np.float32))
    assert ix.sphere_gather((0, 0, 0), 5.0).size == 0


def test_clearance_flat_path_equals_warp_per_trajectory_path(ix, tmp_path):
    """The flat path (schedule / eval / finish kernels) and the one-warp-per-trajectory kernel (PC_CLEARANCE_FLAT=0, also the
    path for schedules beyond 2^27 samples) return identical arrays; the latter runs in a subprocess (the switch is read once)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {root!r})\n"
        "from pointcloudtraj_b200 import PcRadiusParams, PointCloudIndex, synth\n"
        "pts, half = synth.forest_cloud(150_000, seed=6, variant='J', return_half=True)\n"
        "tr = synth.bezier_trajectories(700, half * 0.9, seed=9)\n"
        "tn = np.where(np.arange(700) % 3 == 0, 0.7, 0.0)\n"
        "P = PcRadiusParams.make(0.25, 1.5, 30.0, (0.0, 0.0, 2.0))\n"
        "ix = PointCloudIndex(max_points=len(pts), device=0); ix.build(pts)\n"
        "fh, mr, ns = ix.clearance(tr['traj_first_seg'], tr['seg_order'], tr['seg_T'], tr['seg_coef_off'], tr['coef'], P, t_now=tn, dt=0.02, horizon=7.0)\n"
        "np.savez(sys.argv[1], fh=fh, mr=mr, ns=ns)\n")
    outs = []
    for flat in ("1", "0"):
        path = str(tmp_path / f"clr{flat}.npz")
        env = dict(os.environ, PC_CLEARANCE_FLAT=flat)
        p = subprocess.run([sys.executable, "-c", code, path], env=env, capture_output=True, text=True, timeout=300)
        assert p.returncode == 0, p.stderr
        outs.append(np.load(path))
    a, b = outs
    assert (a["ns"] == b["ns"]).all() and (a["fh"] == b["fh"]).all() and (a["mr"] == b["mr"]).all()
    assert a["ns"].max() > 300 and (a["fh"] >= 0).any() and (a["fh"] < 0).any()
