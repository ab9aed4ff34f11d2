"""Every route of pc_nearest_batch / pc_radius_batch against the CPU kd-tree.

A batch reaches one of many kernels and orderings (pc_query_dispatch, pc_run_batch): the memory space, the batch size against
the tiny / lane-group / ordering / chunk thresholds, the flags, the batch's density (queries per cell of 1/256 of the cloud's
extent: 64-query packets from 3, the 32-bit order above 16) and the PC_* switches read at pc_index_create.  Four datasets reach
them:

1. mid: a 200 k-point jittered forest and a 700 k-query batch with exact cloud points, queries at 1e6 m, NaN / +-inf rows and
   queries beyond the sensing range spliced in at the size thresholds; its prefixes straddle every threshold;
2. bench: bench.py's rank-0 batch, 10 M queries on the 1 M-point map (cell binning + 64-query packets, deferred packets);
3. dense: a flat lattice (the ground caps of a lattice forest) with half of the queries snapped to the lattice (exact ties),
   dense enough for 64-query packets at 400 k queries and for the 32-bit order at 1.5 M, and a two-cluster batch whose
   packets across the gap are put aside;
4. tiny: a collinear lattice, where a few thousand queries are already dense, checked row by row against the brute force.

Each dataset's reference answers are its PC_QUERY_UNSORTED PC_DEVICE results (the thread-per-query kernel), themselves checked
against the CPU kd-tree (tests/parity.py tie rule), its radiusSearch and a numpy restatement of the radius epilogue; every other
route must return the same bits on every row, non-finite rows included.
"""
import ctypes as C

import numpy as np
import pytest

import oracle
from parity import check_lowest_index_everywhere, check_nearest
from pointcloudtraj_b200 import (PC_ARITH_PCL_FLOAT, PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED, PC_RADIUS_BOUNDED,
                                 PC_RADIUS_FULL_NN, PcError, PcRadiusParams, PcSampler, PointCloudIndex, synth)
from pointcloudtraj_b200 import _lib as L

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

CLEAN = dict(search_margin=0.25, max_radius=1.5, sample_range=30.0)      # bench.py's parameters
START = (0.0, 0.0, 2.0)
P = PcRadiusParams.make(start=START, **CLEAN)
OP = oracle.RadiusParams.make(start=START, **CLEAN)
KINDS = ("nearest", "bounded", "full")
NOT_MINE = PointCloudIndex.NOT_MINE_IDX

# prefixes of the mid batch: around PC_TINY_BATCH (4096), the lane-group widths (6144, 12288), PC_COOP_MAX_BATCH (24576) and its
# unbounded form (8192), PC_SORT_MIN_NEAREST (360000), PC_SORT_MIN_RADIUS (640000), and the packet sizes (32, 64)
MID_SIZES = [1, 31, 32, 33, 63, 64, 65, 4096, 4097, 6144, 6145, 8192, 8193, 12288, 12289, 24576, 24577,
             359_999, 360_000, 360_001, 639_999, 640_000, 640_001, 700_000]

# one handle per switch; each is read once, at pc_index_create
SWITCHES = [
    # 32-query packets on the dense batches too, 64-query packets on the sparse ones
    {"PC_QUERY_KERNEL": 3}, {"PC_QUERY_KERNEL": 4},
    # 24 bits: cell binning (bounded radius) and the 24-bit radix order on batches dense enough for 32 bits
    {"PC_SORT_BITS": 0}, {"PC_SORT_BITS": 16}, {"PC_SORT_BITS": 24}, {"PC_SORT_BITS": 32},
    {"PC_BIN_BITS": 12}, {"PC_BIN_BITS": 24},
    {"PC_ONESWEEP": 0},
    {"PC_PACKET_SPLIT": 0}, {"PC_PACKET_SPLIT": 0.5},
    # one lane-group width for every small unordered batch
    {"PC_COOP_GROUP": 32}, {"PC_COOP_GROUP": 16}, {"PC_COOP_GROUP": 8},
    {"PC_COOP_MAX_BATCH": 0}, {"PC_COOP_MAX_BATCH": 1 << 30},
    {"PC_SORT_MIN_BATCH": 1},
    # small blocking PC_HOST calls through the staged pipeline: always, and above 64 queries (the mid sizes straddle 64)
    {"PC_TINY_BATCH_QUERIES": 0}, {"PC_TINY_BATCH_QUERIES": 64},
    {"PC_HOST_CHUNK_QUERIES": 1024},
    # the 700 k batch in a 524 288-query chunk and a 175 712-query tail: the first chunk is above PC_SORT_MIN_NEAREST and below
    # PC_SORT_MIN_RADIUS, so the chunks of one call take different paths
    {"PC_HOST_CHUNK_QUERIES": 1 << 19},
]


def _sid(env):
    return ",".join(f"{k}={v}" for k, v in env.items())


# ---- helpers --------------------------------------------------------------------------------------------------------------
def make_handle(env=None, max_points=0):
    """A handle created under the PC_* environment `env` (read once, at create; the process environment is restored)."""
    with pytest.MonkeyPatch.context() as mp:
        for k, v in (env or {}).items():
            mp.setenv(k, str(v))
        return PointCloudIndex(max_points=max_points, device=0)


def build(h, pts):
    """Build and wait: the density estimate reads the host copy of the bounding box, without which a batch silently takes the
    sparse path."""
    h.build(pts)
    h.sync()
    return h


def per_cell(pts, m):
    """Restatement of the density estimate of the ordering step (pc_order_batch in pc_index.cu): queries per cell of 1/256 of
    the cloud's largest extent, with thin axes counted as one cell.  pc_run_batch takes 64-query packets from 3, and the
    ordering pass the 32-bit order above 16."""
    ext = (pts.max(0) - pts.min(0)).astype(np.float32)
    cell = float(ext.max()) / 256.0
    vol = float(np.prod([max(float(e), cell) for e in ext]))
    return m * cell ** 3 / vol


def _np(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def same(a, b):
    """Bit equality (NaN payloads included)."""
    a, b = _np(a), _np(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def differ(got, want, rows=None):
    """Failure message: how many entries differ, and the first few (row, got, want)."""
    got, want = _np(got), _np(want)
    if got.shape != want.shape:
        return f"shape {got.shape} vs {want.shape}"
    bad = np.nonzero(got.view(np.uint32) != want.view(np.uint32))[0]
    at = bad[:4] if rows is None else np.asarray(rows)[bad[:4]]
    return f"{bad.size} of {got.size} differ, first rows {at.tolist()}: {got[bad[:4]].tolist()} vs {want[bad[:4]].tolist()}"


def run(h, q, kind, space="host", flags=PC_QUERY_AUTO):
    """-> (idx, d2) for nearest, (radius, idx) for the radius kinds, as numpy arrays."""
    if space == "stride4":
        q = np.concatenate([q, np.ones((len(q), 1), np.float32)], 1)
    elif space == "device":
        q = torch.from_numpy(q).cuda()
    if kind == "nearest":
        a, b = h.nearest(q, flags=flags)
    else:
        a, b = h.radius(q, P, flags=(PC_RADIUS_FULL_NN if kind == "full" else PC_RADIUS_BOUNDED) | flags, want_idx=True)
    return _np(a), _np(b)


def run_async(h, qs, kind, space, shard=False):
    """PC_HOST_ASYNC (pinned host buffers) or PC_DEVICE_ASYNC: all batches of `qs` in flight at once, each with its own
    buffers, one wait.  shard: outputs pre-filled as the wrapper does for pc_batch_shard handles."""
    pin = space == L.PC_HOST_ASYNC
    keep = []
    torch.cuda.synchronize()
    for q in qs:
        tq = torch.from_numpy(q).pin_memory() if pin else torch.from_numpy(q).cuda()
        dev = "cpu" if pin else "cuda"
        ti = torch.full((len(q),), NOT_MINE if shard else -7, dtype=torch.int32, device=dev)
        tf = torch.full((len(q),), float("nan") if shard else -7.0, dtype=torch.float32, device=dev)
        if pin:
            ti, tf = ti.pin_memory(), tf.pin_memory()
        vp = lambda t: C.c_void_p(t.data_ptr())
        if kind == "nearest":
            rc = h._L.pc_nearest_batch(h._h, vp(tq), len(q), 3, space, 0, vp(ti), vp(tf))
        else:
            fl = PC_RADIUS_FULL_NN if kind == "full" else PC_RADIUS_BOUNDED
            rc = h._L.pc_radius_batch(h._h, vp(tq), len(q), 3, space, fl, C.byref(P), vp(tf), vp(ti))
        assert rc == 0, h._L.pc_last_error(h._h).decode()
        keep.append((tq, ti, tf))
    h.sync()
    torch.cuda.synchronize()
    return [(ti.cpu().numpy(), tf.cpu().numpy()) if kind == "nearest" else (tf.cpu().numpy(), ti.cpu().numpy())
            for _, ti, tf in keep]


def radius_expect(pts, q, nn, pcl=False):
    """The radiusSearch epilogue (corridor_finder.cpp:113-133) restated on the nearest point nn of every (finite) query:
    sqrt(d2) - margin clamped to max_radius, max_radius - margin beyond the sensing range.  pcl: PC_ARITH_PCL_FLOAT (d2 rounded
    to float32, float32 sqrt, double subtraction).  Returns the double value; the call writes it rounded to float32."""
    d2 = oracle.pair_d2(pts, q, nn.astype(np.int64))
    root = np.sqrt(d2.astype(np.float32)).astype(np.float64) if pcl else np.sqrt(d2)
    r = np.minimum(root - CLEAN["search_margin"], CLEAN["max_radius"])
    r[_far(q)] = CLEAN["max_radius"] - CLEAN["search_margin"]
    return r


def _far(q):
    return np.sqrt(((q.astype(np.float64) - np.array(START)) ** 2).sum(1)) > CLEAN["sample_range"] + CLEAN["max_radius"]


class Dataset:
    """A cloud, a batch, and the batch's reference answers: the PC_QUERY_UNSORTED PC_DEVICE results of a default handle,
    checked against the CPU kd-tree (`rows`: the rows checked, all finite rows by default) before any test uses them."""

    def __init__(self, h, pts, q, tie_free, rng, rows=None, radius_rows=30_000):
        self.pts, self.q, self.h = pts, q, h
        build(h, pts)
        self.base = {k: run(h, q, k, "device", PC_QUERY_UNSORTED) for k in KINDS}
        finite = np.isfinite(q).all(1)
        self.nan = np.isnan(q).any(1)
        fin = np.nonzero(finite)[0]
        rows = fin if rows is None else rng.choice(fin, min(rows, len(fin)), replace=False)
        self.ko = oracle.KdOracle().build(pts, np.random.default_rng(0).permutation(len(pts)))
        idx, d2 = self.base["nearest"]
        ridx, rd2 = self.ko.nearest(q[rows])
        check_nearest(pts, q[rows], idx[rows], d2[rows], ridx, rd2)
        assert (idx[self.nan] == -1).all(), "a NaN query has no neighbour"
        assert (idx[fin] >= 0).all()
        # the radius epilogue of the nearest distance, on every finite row
        expect = radius_expect(pts, q[fin], idx[fin])
        far = _far(q[fin])
        clamped = ~(expect < CLEAN["max_radius"])
        for kind in ("bounded", "full"):
            r, ri = self.base[kind]
            assert same(r[fin], expect.astype(np.float32)), f"{kind} radius: " + differ(r[fin], expect.astype(np.float32), fin)
            assert (ri[self.nan] == -1).all(), kind
            want = idx[fin].copy()
            if kind == "bounded":
                want[clamped] = -1                        # nothing within max_radius + margin: no index
            assert same(ri[fin][~far], want[~far]), f"{kind} index: " + differ(ri[fin][~far], want[~far], fin[~far])
        # the CPU radiusSearch on a sample
        sub = rng.choice(fin, min(radius_rows, len(fin)), replace=False)
        rr, rri = self.ko.radius_batch(OP, q[sub])
        for kind in ("bounded", "full"):
            assert same(self.base[kind][0][sub], rr.astype(np.float32)), f"{kind} vs radiusSearch: " + differ(self.base[kind][0][sub], rr.astype(np.float32), sub)
        if tie_free:
            assert (self.base["full"][1][sub] == rri).all()
        self.fin = fin

    def want(self, kind, m=None):
        a, b = self.base[kind]
        return (a, b) if m is None else (a[:m], b[:m])


def check_prefixes(h, ds, sizes, kinds=KINDS, flags=(PC_QUERY_AUTO, PC_QUERY_SORTED), spaces=("host",)):
    for m in sizes:
        for kind in kinds:
            want = ds.want(kind, m)
            for fl in flags:
                for sp in spaces:
                    got = run(h, ds.q[:m], kind, sp, fl)
                    assert same(got[0], want[0]) and same(got[1], want[1]), \
                        f"{kind}, {m} queries, flags {fl}, {sp}: " + differ(got[0], want[0]) + "; " + differ(got[1], want[1])


def check_async(h, ds, m=None, kinds=KINDS):
    """Three batches in flight in each ASYNC space: the batch, its reverse and a rotation, each with its own buffers."""
    q = ds.q[:m] if m else ds.q
    n = len(q)
    perms = [np.arange(n), np.arange(n)[::-1].copy(), np.roll(np.arange(n), n // 3)]
    for space in (L.PC_HOST_ASYNC, L.PC_DEVICE_ASYNC):
        for kind in kinds:
            want = ds.want(kind, n)
            outs = run_async(h, [np.ascontiguousarray(q[p]) for p in perms], kind, space)
            for p, got in zip(perms, outs):
                assert same(got[0], want[0][p]) and same(got[1], want[1][p]), f"{kind}, space {space}"


def launches_of(h, fn):
    n0 = h.launches()
    fn()
    return h.launches() - n0


def deferred_packets(h):
    d = C.c_int64(-1)
    assert h._L.pc_profile_last_deferred_packets(h._h, C.byref(d)) == 0
    return d.value


def shard_check(h, ds, kind, space, n_ranks, m=None):
    """pc_batch_shard emulated on one handle: every rank gets the same batch; every query must be answered by exactly one rank,
    with the unsharded answer."""
    q = ds.q if m is None else ds.q[:m]
    want = ds.want(kind, len(q))
    owners = np.zeros(len(q), np.int32)
    got = [np.full(len(q), -9, want[0].dtype), np.full(len(q), -9, want[1].dtype)]
    try:
        for r in range(n_ranks):
            h.batch_shard(r, n_ranks)
            if space in ("host", "device"):
                a, b = run(h, q, kind, space)
            else:
                (a, b), = run_async(h, [q], kind, space, shard=True)
            idx = a if kind == "nearest" else b
            mine = idx != NOT_MINE
            owners += mine
            got[0][mine], got[1][mine] = a[mine], b[mine]
    finally:
        h.batch_shard(0, 1)
    assert (owners == 1).all(), f"{kind}, {space}: {(owners != 1).sum()} queries not owned by exactly one rank"
    assert same(got[0], want[0]) and same(got[1], want[1]), f"{kind}, {space}"


# ---- datasets -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def h0():
    h = make_handle()
    yield h
    h.close()


@pytest.fixture(scope="module")
def mid(h0):
    pts, half = synth.forest_cloud(200_000, seed=6, variant="J", return_half=True)
    q = synth.rrt_queries(700_000, half, seed=21)
    rng = np.random.default_rng(21)
    # special rows at both sides of every prefix boundary, so that each prefix ends on one and the next size begins with one
    at = sorted({b for m in MID_SIZES for b in (m - 1, m) if b < len(q)})
    special = [
        lambda: pts[rng.integers(len(pts))],                        # exactly a cloud point
        lambda: np.array([1e6, -1e6, 3.0], np.float32),              # a million metres away
        lambda: np.array([np.nan, 1.0, 2.0], np.float32),
        lambda: np.array([np.inf, 0.0, 2.0], np.float32),
        lambda: np.array([0.0, -np.inf, 2.0], np.float32),
        lambda: np.array([40.0, 5.0, 2.0], np.float32),              # beyond the sensing range (sample_range + max_radius)
        lambda: np.array([1.0, np.nan, np.nan], np.float32),
    ]
    for k, row in enumerate(at):
        q[row] = special[k % len(special)]()
    ds = Dataset(h0, pts, q, tie_free=True, rng=rng)
    assert per_cell(pts, len(q)) < 3.0, "the mid batch is sparse: 32-query packets"
    return ds


@pytest.fixture(scope="module")
def bench_ds(h0):
    """bench.py's rank-0 step: the 1 M-point map (seed 1) and rrt_queries(10 M, half, seed=1000)."""
    pts, half = synth.forest_cloud(1_000_000, seed=1, variant="J", return_half=True)
    q = synth.rrt_queries(10_000_000, half, seed=1000)
    return Dataset(h0, pts, q, tie_free=True, rng=np.random.default_rng(5), rows=300_000)


def _flat_lattice():
    pts, half = synth.forest_cloud(200_000, seed=6, variant="L", return_half=True)
    return np.ascontiguousarray(pts[pts[:, 2] == 0]), half


@pytest.fixture(scope="module")
def dense(h0):
    """Flat lattice (ground caps of a lattice forest), 1.5 M queries near the plane, half of them snapped to the lattice."""
    pts, half = _flat_lattice()
    q = synth.rrt_queries(1_500_000, half, seed=31, z=(-0.3, 0.3), lattice_frac=0.5)
    rng = np.random.default_rng(31)
    q[rng.choice(len(q), 2000, replace=False)] = pts[rng.integers(len(pts), size=2000)]
    ds = Dataset(h0, pts, q, tie_free=False, rng=rng, rows=300_000)
    assert 4.0 < per_cell(pts, 400_000) < 12.0, "400 k queries: 64-query packets, 24-bit order"
    assert per_cell(pts, len(q)) > 20.0, "1.5 M queries: 32-bit order"
    return ds


@pytest.fixture(scope="module")
def two_clusters(h0):
    """Queries in two boxes at opposite corners of the flat lattice: the curve order jumps between them, so packets across
    the jumps hold queries tens of metres apart and the unbounded walks put them aside."""
    pts, half = _flat_lattice()
    rng = np.random.default_rng(41)
    n = 200_003                                        # not a multiple of the packet size
    a = rng.uniform([-half, -half, -0.3], [-half / 2, -half / 2, 0.3], (n, 3))
    b = rng.uniform([half / 2, half / 2, -0.3], [half, half, 0.3], (n, 3))
    q = np.concatenate([a, b]).astype(np.float32)
    q = np.ascontiguousarray(q[rng.permutation(len(q))])
    q[::2] = np.round(q[::2] / 0.05) * 0.05
    ds = Dataset(h0, pts, q, tie_free=False, rng=rng, rows=100_000, radius_rows=10_000)
    assert 4.0 < per_cell(pts, len(q)) < 12.0
    return ds


# ---- the default handle ---------------------------------------------------------------------------------------------------
def test_mid_every_size_and_space(h0, mid):
    build(h0, mid.pts)
    check_prefixes(h0, mid, MID_SIZES, flags=(PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED), spaces=("host", "stride4", "device"))
    check_async(h0, mid)
    check_async(h0, mid, m=4097)


def test_bench_batch(h0, bench_ds):
    """bench.py's batch: bounded radius through the cell binning and 64-query packets, nearest and FULL_NN through the 24-bit
    radix order, 64-query packets and the deferred kernel; PC_HOST as ten pipelined chunks (the last, 562 816 queries, is
    too small to be ordered for radius but not for nearest)."""
    ds, h = bench_ds, h0
    build(h, ds.pts)
    pc = per_cell(ds.pts, len(ds.q))
    assert 4.0 < pc < 12.0 and per_cell(ds.pts, 1 << 20) < 3.0
    for kind in KINDS:
        got = []
        n = launches_of(h, lambda: got.append(run(h, ds.q, kind, "device")))
        # cell binning (5 kernels) + search for bounded radius; key kernel + 3 onesweep passes + search + deferred for the others
        assert n == 6, (kind, n)
        assert same(got[0][0], ds.want(kind)[0]) and same(got[0][1], ds.want(kind)[1]), kind
        got = run(h, ds.q, kind, "host")
        assert same(got[0], ds.want(kind)[0]) and same(got[1], ds.want(kind)[1]), kind
    check_async(h, ds, kinds=("nearest", "bounded"))


def test_dense_ties(h0, dense):
    ds, h = dense, h0
    build(h, ds.pts)
    sizes = [64, 4097, 100_000, 400_000, 1 << 20, (1 << 20) + 1, 1_500_000]
    check_prefixes(h, ds, sizes, spaces=("host", "device"))
    # the observable of each ordering (sorted batches): 24-bit radix (key kernel + 3 passes) + search + deferred = 6, 32-bit = 7;
    # cell binning for bounded radius at 24 bits = 5 + search; 32-bit radix for bounded radius = 1 + 4 + search, no deferral
    expect = {("nearest", 400_000): 6, ("nearest", 1_500_000): 7, ("bounded", 400_000): 6, ("bounded", 1_500_000): 6,
              ("full", 400_000): 6, ("full", 1_500_000): 7}
    for (kind, m), n in expect.items():
        assert launches_of(h, lambda: run(h, ds.q[:m], kind, "device", PC_QUERY_SORTED)) == n, (kind, m)
    # unordered: one search kernel (a bounded batch below PC_SORT_MIN_RADIUS, 640 000, is not ordered by default)
    assert launches_of(h, lambda: run(h, ds.q[:400_000], "nearest", "device", PC_QUERY_UNSORTED)) == 1
    assert launches_of(h, lambda: run(h, ds.q[:400_000], "bounded", "device")) == 1
    check_async(h, ds, m=400_000)
    # PC_HOST one query above a chunk: an ordered 2^20 chunk and a one-query tail
    for kind in KINDS:
        got = run(h, ds.q[:(1 << 20) + 1], kind, "host")
        want = ds.want(kind, (1 << 20) + 1)
        assert same(got[0], want[0]) and same(got[1], want[1])


def test_two_cluster_packets_are_deferred(h0, two_clusters):
    ds, h = two_clusters, h0
    build(h, ds.pts)
    for kind in ("nearest", "full"):
        got = run(h, ds.q, kind, "device", PC_QUERY_SORTED)
        assert deferred_packets(h) >= 1, kind
        assert same(got[0], ds.want(kind)[0]) and same(got[1], ds.want(kind)[1]), kind
        got = run(h, ds.q, kind, "host")
        assert same(got[0], ds.want(kind)[0]) and same(got[1], ds.want(kind)[1]), kind
    got = run(h, ds.q, "bounded", "host")
    assert same(got[0], ds.want("bounded")[0]) and same(got[1], ds.want("bounded")[1])


@pytest.mark.parametrize("m", [2000, 8000])
def test_tiny_dense_collinear(h0, m):
    """A collinear lattice with duplicate points: per_cell = m / 256, so 2000 sorted queries take 64-query packets and 8000
    the 32-bit order.  Every row against the brute force (lowest index among exact ties)."""
    rng = np.random.default_rng(m)
    pts = np.zeros((3000, 3), np.float32)
    pts[:, 0] = np.round(rng.uniform(-50, 50, len(pts)) / 0.1) * 0.1
    q = np.zeros((m, 3), np.float32)
    q[:, 0] = rng.uniform(-55, 55, m)
    q[:, 1:] = rng.uniform(-0.5, 0.5, (m, 2))
    q[::2, 0] = np.round(q[::2, 0] / 0.05) * 0.05          # midway between two lattice points, or on one
    q[::4, 1:] = 0.0
    assert (4.0 < per_cell(pts, m) < 12.0) if m == 2000 else per_cell(pts, m) > 20.0
    h = build(h0, pts)
    bi, bd, _ = oracle.brute_nearest(pts, q)
    r64 = radius_expect(pts, q, bi)
    expect_r = r64.astype(np.float32)
    for space in ("host", "device"):
        idx, d2 = run(h, q, "nearest", space, PC_QUERY_SORTED)
        check_lowest_index_everywhere(pts, q, idx)
        assert (d2 == bd.astype(np.float32)).all()
        for kind in ("bounded", "full"):
            r, ri = run(h, q, kind, space, PC_QUERY_SORTED)
            assert same(r, expect_r), kind
            near = ~_far(q)
            want = bi.copy()
            if kind == "bounded":
                want[~(r64 < CLEAN["max_radius"])] = -1
            assert (ri[near] == want[near]).all(), kind
    n = launches_of(h, lambda: run(h, q, "nearest", "device", PC_QUERY_SORTED))
    assert n == (6 if m == 2000 else 7)


# ---- every switch -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env", SWITCHES, ids=_sid)
def test_switch_mid(mid, env):
    h = make_handle(env)
    try:
        build(h, mid.pts)
        chunked = "PC_HOST_CHUNK_QUERIES" in env
        sizes = [1, 33, 65, 4097, 24577, 360_001, 700_000] if chunked else MID_SIZES
        check_prefixes(h, mid, sizes)
        check_prefixes(h, mid, [700_000], flags=(PC_QUERY_AUTO,), spaces=("device",))
    finally:
        h.close()


@pytest.mark.parametrize("env", SWITCHES, ids=_sid)
def test_switch_dense(dense, two_clusters, env):
    h = make_handle(env)
    try:
        build(h, dense.pts)
        check_prefixes(h, dense, [400_000, 1_500_000], flags=(PC_QUERY_AUTO,), spaces=("host", "device"))
        for kind in ("nearest", "full"):
            for sp in ("host", "device"):
                got = run(h, two_clusters.q, kind, sp, PC_QUERY_SORTED)
                assert same(got[0], two_clusters.want(kind)[0]) and same(got[1], two_clusters.want(kind)[1]), (kind, sp)
    finally:
        h.close()


# ---- PC_ARITH_PCL_FLOAT -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["mid", "bench"])
def test_pcl_float_arithmetic(request, which):
    ds = request.getfixturevalue("mid" if which == "mid" else "bench_ds")
    h = build(make_handle(), ds.pts)
    try:
        h.set_radius_arith(PC_ARITH_PCL_FLOAT)
        idx = ds.want("nearest")[0]
        r64 = radius_expect(ds.pts, ds.q[ds.fin], idx[ds.fin], pcl=True)
        expect = r64.astype(np.float32)
        # a bounded search reports no index where the radius clamps, and the clamp is decided in the chosen arithmetic
        near = ~_far(ds.q[ds.fin])
        want_idx = {"full": ds.want("full")[1], "bounded": ds.want("bounded")[1].copy()}
        want_idx["bounded"][ds.fin[near]] = np.where(r64[near] < CLEAN["max_radius"], idx[ds.fin[near]], -1)
        spaces = ("host", "device") if which == "mid" else ("device",)
        for kind in ("bounded", "full"):
            for sp in spaces:
                for fl in (PC_QUERY_AUTO, PC_QUERY_UNSORTED):
                    r, ri = run(h, ds.q, kind, sp, fl)
                    assert same(r[ds.fin], expect), f"{kind} {sp} {fl}: " + differ(r[ds.fin], expect, ds.fin)
                    assert same(ri, want_idx[kind]), f"{kind} {sp} {fl}: " + differ(ri, want_idx[kind])
                    nf = np.ones(len(ds.q), bool)
                    nf[ds.fin] = False
                    assert same(r[nf], ds.want(kind)[0][nf])
        assert not same(expect, ds.want("full")[0][ds.fin]), "the two arithmetics differ somewhere on this batch"
    finally:
        h.close()


# ---- pc_batch_shard -----------------------------------------------------------------------------------------------------
def test_shard_bench(bench_ds):
    ds = bench_ds
    h = build(make_handle(), ds.pts)
    h_nx = build(make_handle({"PC_SHARD_EXACT": 0}), ds.pts)
    try:
        for kind in KINDS:
            shard_check(h, ds, kind, "device", 3)          # bins (bounded) / radix (others), share size read back
            shard_check(h_nx, ds, kind, "device", 2)       # launches sized for the whole batch
            shard_check(h, ds, kind, "host", 2)            # ten pipelined chunks
            shard_check(h, ds, kind, L.PC_HOST_ASYNC, 2)
    finally:
        h.close()
        h_nx.close()


def test_shard_dense(dense):
    ds = dense
    h = build(make_handle(), ds.pts)
    h_nx = build(make_handle({"PC_SHARD_EXACT": 0}), ds.pts)
    h_ch = build(make_handle({"PC_HOST_CHUNK_QUERIES": 1024}), ds.pts)
    try:
        for kind in KINDS:
            shard_check(h, ds, kind, "device", 3)                      # 32-bit order, share size read back
            shard_check(h, ds, kind, "device", 2, m=400_000)            # bins (bounded) / 24-bit radix
            shard_check(h_nx, ds, kind, "device", 2)
            shard_check(h, ds, kind, L.PC_HOST_ASYNC, 2, m=400_000)
            shard_check(h_ch, ds, kind, "host", 2, m=200_000)           # 196 chunks of 1024 queries
    finally:
        h.close()
        h_nx.close()
        h_ch.close()


# ---- pc_expand_batch ----------------------------------------------------------------------------------------------------
def test_expand_batch_refuses_sharded_handles(mid):
    """pc_expand_batch needs the radius of every centre and the nearest vertex of every sample: a pc_batch_shard handle on
    either side is refused before anything runs, and both handles work again once sharding is switched off."""
    start, end, box = (0.0, 0.0, 2.0), (40.0, 10.0, 2.0), (-50.0, 50.0, -50.0, 50.0, 0.0, 5.0)
    rng = np.random.default_rng(3)
    n_nodes, k = 37, 4096                            # small enough for the brute-force nearest vertex
    node_coord = np.column_stack([rng.uniform(-25, 25, n_nodes), rng.uniform(-25, 25, n_nodes), rng.uniform(0.7, 4.0, n_nodes)])
    node_coord[0] = start
    node_radius = rng.uniform(0.6, 1.25, n_nodes).astype(np.float32)
    node_valid = np.ones(n_nodes, np.uint8)
    sampler = lambda: PcSampler.make(start, end, box, 30.0, 0.6, 0.3, 0.15, engine_state=777)
    cloud = build(make_handle(), mid.pts)
    nodes = make_handle()
    try:
        expand = lambda s: cloud.expand_batch(nodes, node_coord, node_radius, node_valid, s, P, box[4], 0.6, k)
        want = expand(sampler())
        assert len(want) > 0
        for sharded in (cloud, nodes):
            sharded.batch_shard(1, 2)
            s = sampler()
            try:
                with pytest.raises(PcError) as e:
                    expand(s)
                assert e.value.code == L.PC_EINVAL and "pc_batch_shard" in str(e.value)
                assert s.engine_state == 777
            finally:
                sharded.batch_shard(0, 1)
            got = expand(sampler())
            assert (got == want).all()
    finally:
        cloud.close()
        nodes.close()
