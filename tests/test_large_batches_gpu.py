"""Every batch call past 2^30 rows, 2^31 output entries and 2^32 voxels, against sub-batch runs and the fp64 references.

The C ABI takes up to 2^32 - 1 rows per call, int64 CSR offsets and up to 2^40 voxels, and several code paths only run at such
sizes: the ordering sort leaves the fused onesweep histograms at 2^30 entries (OS_MAX_N), bounded radius batches stop binning
at 2^32 - 1 rows, and the row x k, CSR and voxel stores pass 2^31 and 2^32 entries.  A 32-bit product that wraps there, or a
counter that saturates, leaves every smaller batch right.  Each case below therefore runs one batch across such a boundary
and checks it twice:

1. every row against the same call run as consecutive sub-batches of < 2^28 rows (< 2^31 output entries) -- pointers offset
   into the same device tensors, so the sub-batches take the paths the rest of the suite covers.  Rows are independent under
   the exactness contract, so the outputs must be bit-identical; CSR rows are compared by length and by entries with each
   sub-batch's offsets shifted;
2. about 10^5 sampled rows -- the first and last 4096, +-4096 around every boundary row, random rows -- against the fp64
   references (CPU kd-tree, brute force), which share no code with the library.

One 200 k-point jittered forest is the cloud; queries are made on the device from a seeded generator, with exact cloud points,
NaN / +-inf rows, rows 10^6 m away and rows beyond the radius search's sensing range planted at and just past every boundary.

Memory: each case's estimate (the _budget call, its terms commented) is checked against torch.cuda.mem_get_info() after the index is built, with 15 %
head-room; a case that does not fit at its size is skipped with the bytes it needed (a smaller size would not cross its
boundary).  The library's buffers come from the device's default memory pool, which keeps freed memory (pc_pool_setup), so
after every case the handle is destroyed, the pool trimmed and torch's cache emptied.  Both outputs of a nearest batch of
2^32 - 1 rows (about 164 GB with the queries and sort buffers) do not fit a 180 GB device with that head-room, so the
nearest and bounded radius cases at 2^32 - 1 rows write one output each.
"""
import contextlib
import ctypes as C
import gc

import numpy as np
import pytest

import oracle
from knn_brute import brute_knn
from parity import check_nearest
from range_sorted_brute import brute_range_sorted
from segment_brute import brute_segment
from sweep_brute import brute_sweep, round_down_f32
from pointcloudtraj_b200 import (PC_QUERY_SORTED, PC_RADIUS_BOUNDED, PC_RADIUS_FULL_NN, PcRadiusParams, PointCloudIndex,
                                 synth)
from pointcloudtraj_b200 import _lib as L

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

G = 1 << 30
SUB = 1 << 27                # rows per sub-batch: fused onesweep, cell binning, < 2^31 entries at k <= 4
W = 4096                     # rows sampled on each side of a boundary
HEADROOM = 1.15
CLEAN = dict(search_margin=0.25, max_radius=1.5, sample_range=30.0)
START = (0.0, 0.0, 2.0)
P = PcRadiusParams.make(start=START, **CLEAN)
OP = oracle.RadiusParams.make(start=START, **CLEAN)
SEG_RANGE = 2.0
SWEEP_R = 0.3
KNN_R = 1.0
FIELD_R = 1.0


def _vp(t):
    return C.c_void_p(t.data_ptr())


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _release():
    """Give the device back between cases: torch's cache and the library's memory pool (which never trims itself)."""
    torch.cuda.synchronize()
    gc.collect()
    torch.cuda.empty_cache()
    cu = C.CDLL("libcuda.so.1")
    dev, pool = C.c_int(0), C.c_void_p()
    assert cu.cuDeviceGet(C.byref(dev), torch.cuda.current_device()) == 0
    assert cu.cuDeviceGetDefaultMemPool(C.byref(pool), dev) == 0
    assert cu.cuMemPoolTrimTo(pool, C.c_size_t(0)) == 0


def _budget(need, what):
    free = torch.cuda.mem_get_info()[0]
    if need * HEADROOM > free:
        pytest.skip(f"{what}: needs {need} bytes of device memory + 15 % head-room, {free} free")
    print(f"\n{what}: about {need / 1e9:.1f} GB of {free / 1e9:.1f} GB free")


def _host_budget(need, what):
    avail = 0
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    if need * HEADROOM > avail:
        pytest.skip(f"{what}: needs {need} bytes of host memory + 15 % head-room, {avail} available")


@pytest.fixture(scope="module")
def cloud():
    pts, half = synth.forest_cloud(200_000, seed=6, variant="J", return_half=True)
    ko = oracle.KdOracle().build(pts, np.random.default_rng(0).permutation(len(pts)))
    return pts, half, ko


@contextlib.contextmanager
def handle(pts, env=None):
    """A handle on torch's stream (calls are ordered with torch work) with the cloud built; destroyed and its memory
    returned to the driver afterwards."""
    _release()
    with pytest.MonkeyPatch.context() as mp:
        for k, v in (env or {}).items():
            mp.setenv(k, str(v))
        h = PointCloudIndex(device=0, stream=torch.cuda.current_stream().cuda_stream)
    try:
        h.build(pts)
        h.sync()
        yield h
    finally:
        h.close()
        _release()


def _ok(h, rc):
    assert rc == L.PC_OK, h._L.pc_last_error(h._h).decode()


# ---- inputs -------------------------------------------------------------------------------------------------------------
def _specials(pts, rng):
    """Rows that take the edges of the search: an exact cloud point (d2 = 0), 10^6 m away, NaN / +-inf, beyond the sensing
    range (the radius early-out)."""
    return np.array([pts[rng.integers(len(pts))], [1e6, -1e6, 3.0], [np.nan, 1.0, 2.0], [np.inf, 0.0, 2.0],
                     [0.0, -np.inf, 2.0], [40.0, 5.0, 2.0], [1.0, np.nan, np.nan], pts[rng.integers(len(pts))]], np.float32)


def _planted_rows(m, boundaries):
    rows = set()
    for b in list(boundaries) + [0, m]:
        rows.update(r for r in range(b - 8, b + 8) if 0 <= r < m)
    return np.array(sorted(rows), np.int64)


def make_queries(m, half, pts, boundaries, seed, z=(0.6, 4.0)):
    """(m, 3) float32 queries on the device, uniform in the map's box, special rows planted around every boundary."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.empty((m, 3), dtype=torch.float32, device="cuda")
    step = 1 << 28
    lo = torch.tensor([-half, -half, z[0]], dtype=torch.float32, device="cuda")
    span = torch.tensor([2 * half, 2 * half, z[1] - z[0]], dtype=torch.float32, device="cuda")
    for off in range(0, m, step):
        blk = q[off:off + step]
        blk.uniform_(0.0, 1.0, generator=gen)
        blk.mul_(span).add_(lo)
    rows = _planted_rows(m, boundaries)
    sp = _specials(pts, np.random.default_rng(seed))
    q[torch.from_numpy(rows).cuda()] = torch.from_numpy(sp[np.arange(len(rows)) % len(sp)]).cuda()
    return q


def sample_rows(m, boundaries, seed, n_random):
    """First and last W rows, +-W around every boundary row, and n_random random rows."""
    parts = [np.arange(0, min(W, m)), np.arange(max(0, m - W), m)]
    for b in boundaries:
        parts.append(np.arange(max(0, b - W), min(m, b + W)))
    parts.append(np.random.default_rng(seed).integers(0, m, n_random))
    rows = np.unique(np.concatenate(parts))
    for b in boundaries:
        assert b - 1 in rows and (b >= m or b in rows), f"boundary row {b} not sampled"
    return rows


def take(t, rows, width=1):
    """Rows of a device tensor (width entries each) as a numpy array."""
    r = torch.from_numpy(rows).cuda()
    if width == 1:
        return t[r].cpu().numpy()
    return t.view(-1, width)[r].cpu().numpy()


# ---- check 1: sub-batches -------------------------------------------------------------------------------------------------
def check_sub_batches(call, m, width, big, sub=SUB, what=""):
    """call(off, c, outs): rows [off, off + c) of the batch into the fresh tensors outs (c * width entries each); big: the
    whole batch's outputs.  Every entry must be bit-identical."""
    n_sub = 0
    for off in range(0, m, sub):
        c = min(sub, m - off)
        outs = [torch.empty(c * width, dtype=b.dtype, device=b.device) for b in big]
        call(off, c, outs)
        for o, b in zip(outs, big):
            s = b[off * width:(off + c) * width]
            if not torch.equal(_bits(o), _bits(s)):
                bad = torch.nonzero(_bits(o) != _bits(s))[:4, 0].cpu().numpy()
                raise AssertionError(f"{what}: rows {(bad // width + off).tolist()} differ from the sub-batch at {off}: "
                                     f"{s[bad].tolist()} vs {o[bad].tolist()}")
        n_sub += 1
        del outs
    assert n_sub >= 2
    return n_sub


# ---- row-per-query calls ------------------------------------------------------------------------------------------------
def nearest_call(h, q, space=L.PC_DEVICE, flags=0):
    def call(off, c, outs):
        d2 = _vp(outs[1]) if len(outs) > 1 else C.c_void_p(0)
        _ok(h, h._L.pc_nearest_batch(h._h, C.c_void_p(q.data_ptr() + off * 12), c, 3, space, flags, _vp(outs[0]), d2))
    return call


def check_nearest_rows(pts, ko, q, idx, d2, rows):
    qs, gi = take(q, rows), take(idx, rows)
    fin = np.isfinite(qs).all(1)
    nan = np.isnan(qs).any(1)
    ri, rd = ko.nearest(qs[fin])
    check_nearest(pts, qs[fin], gi[fin], None if d2 is None else take(d2, rows)[fin], ri, rd)
    assert (gi[nan] == -1).all(), "a NaN query has no neighbour"
    return fin.sum()


@pytest.mark.parametrize("m", [G + 17, 2 * G + 17, 4 * G - 1], ids=["2^30+17", "2^31+17", "2^32-1"])
def test_nearest_device(cloud, m):
    """pc_nearest_batch, PC_DEVICE, PC_QUERY_AUTO: the ordering sort without the fused histograms (m >= 2^30), the uint32
    permutation, the packet and deferred kernels.  At 2^32 - 1 rows (the most one call takes) the index output only: with the
    d2 output the case would not fit 180 GB with the head-room."""
    pts, half, ko = cloud
    bounds = [b for b in (G, 2 * G, 4 * G - 1) if b <= m]
    with_d2 = m < 4 * G - 1
    with handle(pts) as h:
        # queries, outputs, four sort buffers of m words, sort scratch, one sub-batch's outputs
        _budget(m * 12 + m * (8 if with_d2 else 4) + m * 16 + m * 2 + SUB * 8, f"nearest, {m} rows")
        q = make_queries(m, half, pts, bounds, seed=1)
        idx = torch.empty(m, dtype=torch.int32, device="cuda")
        d2 = torch.empty(m, dtype=torch.float32, device="cuda") if with_d2 else None
        big = [idx, d2] if with_d2 else [idx]
        call = nearest_call(h, q)
        call(0, m, big)
        assert m >= G
        check_sub_batches(call, m, 1, big, what="nearest")
        rows = sample_rows(m, bounds, 2, 60_000)
        assert check_nearest_rows(pts, ko, q, idx, d2, rows) > 50_000


def radius_call(h, q, flags, with_idx=True):
    def call(off, c, outs):
        _ok(h, h._L.pc_radius_batch(h._h, C.c_void_p(q.data_ptr() + off * 12), c, 3, L.PC_DEVICE, flags, C.byref(P),
                                    _vp(outs[0]), _vp(outs[1]) if with_idx else C.c_void_p(0)))
    return call


def _far(q):
    return np.sqrt(((q.astype(np.float64) - np.array(START)) ** 2).sum(1)) > CLEAN["sample_range"] + CLEAN["max_radius"]


def check_radius_rows(pts, ko, q, r, rows, idx=None, bounded=True):
    """The radius (and index) of the sampled rows against the CPU radiusSearch and the kd-tree's nearest point."""
    qs, gr = take(q, rows), take(r, rows)
    fin = np.isfinite(qs).all(1)
    rr, _ = ko.radius_batch(OP, qs[fin])
    want = rr.astype(np.float32)
    bad = np.nonzero(gr[fin].view(np.uint32) != want.view(np.uint32))[0]
    assert bad.size == 0, f"{bad.size} radii differ, rows {rows[fin][bad[:4]].tolist()}: {gr[fin][bad[:4]]} vs {want[bad[:4]]}"
    if idx is not None:
        gi = take(idx, rows)
        near = fin & ~_far(qs)
        ni, nd = ko.nearest(qs[near])
        if bounded:
            hit = np.sqrt(nd) - CLEAN["search_margin"] < CLEAN["max_radius"]
            assert (gi[near][~hit] == -1).all(), "bounded: an index beyond max_radius + margin"
            check_nearest(pts, qs[near][hit], gi[near][hit], None, ni[hit], nd[hit])
        else:
            check_nearest(pts, qs[near], gi[near], None, ni, nd)
        assert (gi[np.isnan(qs).any(1)] == -1).all()
    assert _far(qs[fin]).sum() > 0, "no sampled row hit the sensing-range early-out"
    return fin.sum()


@pytest.mark.parametrize("bounded", [True, False], ids=["bounded", "full_nn"])
def test_radius_device(cloud, bounded):
    """pc_radius_batch, PC_DEVICE, 2^30 + 17 rows: the radix order at >= 2^30 rows, early-outs answered by the key kernel."""
    pts, half, ko = cloud
    m = G + 17
    flags = PC_RADIUS_BOUNDED if bounded else PC_RADIUS_FULL_NN
    with handle(pts) as h:
        _budget(m * 12 + m * 8 + m * 16 + m * 2 + SUB * 8, f"radius, {m} rows")
        q = make_queries(m, half, pts, [G], seed=3)
        r = torch.empty(m, dtype=torch.float32, device="cuda")
        idx = torch.empty(m, dtype=torch.int32, device="cuda")
        call = radius_call(h, q, flags)
        call(0, m, [r, idx])
        check_sub_batches(call, m, 1, [r, idx], what="radius")
        rows = sample_rows(m, [G], 4, 60_000)
        assert check_radius_rows(pts, ko, q, r, rows, idx, bounded) > 50_000


def test_radius_bounded_2_32_minus_1(cloud):
    """pc_radius_batch bounded, exactly 2^32 - 1 rows (the most one call takes), 24-bit order: cell binning stops below this
    size, so the batch takes the radix sort; the sub-batches are binned.  Radius output only (an index output would not fit)."""
    pts, half, ko = cloud
    m = (1 << 32) - 1
    with handle(pts, {"PC_SORT_BITS": 24}) as h:
        _budget(m * 12 + m * 4 + m * 16 + m * 2 + SUB * 4 + SUB * 16, f"bounded radius, {m} rows")
        q = make_queries(m, half, pts, [G, 2 * G, 4 * G - 1], seed=5)
        r = torch.empty(m, dtype=torch.float32, device="cuda")
        call = radius_call(h, q, PC_RADIUS_BOUNDED, with_idx=False)
        call(0, m, [r])
        check_sub_batches(lambda off, c, outs: call(off, c, [outs[0], None]), m, 1, [r], what="radius 2^32-1")
        rows = sample_rows(m, [G, 2 * G, 4 * G - 1], 6, 60_000)
        assert check_radius_rows(pts, ko, q, r, rows) > 50_000


def test_nearest_host_chunks(cloud):
    """pc_nearest_batch, PC_HOST on pinned memory (pc_host_alloc), 2^31 + 17 rows: more than 2048 chunks over the pipeline
    lanes, each staged at row off * stride of the caller's arrays.  Checked against PC_DEVICE sub-batches of the same rows."""
    pts, half, ko = cloud
    m = 2 * G + 17
    _host_budget(m * 20, f"PC_HOST nearest, {m} rows")
    with handle(pts) as h:
        _budget(m * 12 + SUB * 16 + (1 << 31), f"PC_HOST nearest, {m} rows")
        hl = h._L
        bufs = [hl.pc_host_alloc(m * 12), hl.pc_host_alloc(m * 4), hl.pc_host_alloc(m * 4)]
        try:
            assert all(bufs)
            hq = np.ctypeslib.as_array(C.cast(bufs[0], C.POINTER(C.c_float)), shape=(m, 3))
            hi = np.ctypeslib.as_array(C.cast(bufs[1], C.POINTER(C.c_int32)), shape=(m,))
            hd = np.ctypeslib.as_array(C.cast(bufs[2], C.POINTER(C.c_float)), shape=(m,))
            q = make_queries(m, half, pts, [G, 2 * G], seed=7)
            torch.from_numpy(hq).copy_(q)
            torch.cuda.synchronize()
            hi[:] = -7
            _ok(h, hl.pc_nearest_batch(h._h, C.c_void_p(bufs[0]), m, 3, L.PC_HOST, 0, C.c_void_p(bufs[1]), C.c_void_p(bufs[2])))
            assert -(-m // (1 << 20)) > 2048
            # every row against PC_DEVICE sub-batches of the device copy of the queries
            call = nearest_call(h, q)
            ti, td = torch.from_numpy(hi), torch.from_numpy(hd)
            for off in range(0, m, SUB):
                c = min(SUB, m - off)
                oi = torch.empty(c, dtype=torch.int32, device="cuda")
                od = torch.empty(c, dtype=torch.float32, device="cuda")
                call(off, c, [oi, od])
                gi, gd = ti[off:off + c].cuda(), td[off:off + c].cuda()
                if not (torch.equal(gi, oi) and torch.equal(_bits(gd), _bits(od))):
                    bad = torch.nonzero((gi != oi) | (_bits(gd) != _bits(od)))[:4, 0].cpu().numpy() + off
                    raise AssertionError(f"PC_HOST rows {bad.tolist()} differ from PC_DEVICE")
            rows = sample_rows(m, [G, 2 * G], 8, 60_000)
            qs = hq[rows]
            fin = np.isfinite(qs).all(1)
            ri, rd = ko.nearest(qs[fin])
            check_nearest(pts, qs[fin], hi[rows][fin], hd[rows][fin], ri, rd)
            assert (hi[rows][np.isnan(qs).any(1)] == -1).all()
            del hq, hi, hd, ti, td
        finally:
            for b in bufs:
                hl.pc_host_free(b)


# ---- kNN ------------------------------------------------------------------------------------------------------------------
def knn_call(h, q, k, r, large=False):
    fn = h._L.pc_knn_large_batch if large else h._L.pc_knn_batch

    def call(off, c, outs):
        _ok(h, fn(h._h, C.c_void_p(q.data_ptr() + off * 12), c, 3, L.PC_DEVICE, 0, k, -1.0 if r is None else r,
                  _vp(outs[0]), _vp(outs[1])))
    return call


def check_knn_rows(pts, q, idx, d2, k, r, rows):
    qs, gi, gd = take(q, rows), take(idx, rows, k), take(d2, rows, k)
    fin = np.isfinite(qs).all(1)
    bi, bd = brute_knn(pts, qs[fin], k, r)
    bad = np.nonzero((gi[fin] != bi).any(1) | (gd[fin] != bd.astype(np.float32)).any(1))[0]
    assert bad.size == 0, f"{bad.size} rows differ from the brute force, first {rows[fin][bad[:4]].tolist()}"
    return fin.sum()


def test_knn_bounded(cloud):
    """pc_knn_batch, k = 4 within 1 m, 2^30 + 17 rows: more than 2^32 output entries (row x k addressing), ordering at
    >= 2^30 rows."""
    pts, half, ko = cloud
    m, k = G + 17, 4
    with handle(pts) as h:
        _budget(m * 12 + m * k * 8 + m * 16 + m * 2 + SUB * k * 8, f"knn k=4, {m} rows")
        q = make_queries(m, half, pts, [G], seed=9)
        idx = torch.empty(m * k, dtype=torch.int32, device="cuda")
        d2 = torch.empty(m * k, dtype=torch.float32, device="cuda")
        call = knn_call(h, q, k, KNN_R)
        call(0, m, [idx, d2])
        assert m * k > 1 << 32
        check_sub_batches(call, m, k, [idx, d2], what="knn")
        # rows whose entries cross 2^31 and 2^32
        rows = sample_rows(m, [G, (1 << 31) // k, (1 << 32) // k], 10, 20_000)
        assert check_knn_rows(pts, q, idx, d2, k, KNN_R, rows) > 20_000


def test_knn_large(cloud):
    """pc_knn_large_batch, k = 1024, 2^21 + 5 rows: more than 2^31 output entries without the big sort."""
    pts, half, ko = cloud
    m, k = (1 << 21) + 5, 1024
    with handle(pts) as h:
        _budget(m * 12 + m * k * 8 * 2, f"knn_large k=1024, {m} rows")
        q = make_queries(m, half, pts, [1 << 21], seed=11)
        idx = torch.empty(m * k, dtype=torch.int32, device="cuda")
        d2 = torch.empty(m * k, dtype=torch.float32, device="cuda")
        call = knn_call(h, q, k, None, large=True)
        call(0, m, [idx, d2])
        assert m * k > 1 << 31
        check_sub_batches(call, m, k, [idx, d2], sub=1 << 19, what="knn_large")
        rows = sample_rows(m, [1 << 21], 12, 2_000)
        assert check_knn_rows(pts, q, idx, d2, k, None, rows) > 10_000


# ---- segments -------------------------------------------------------------------------------------------------------------
def make_segments(m, half, pts, boundaries, seed):
    a = make_queries(m, half, pts, boundaries, seed)
    b = torch.empty_like(a)
    gen = torch.Generator(device="cuda").manual_seed(seed + 1)
    step = 1 << 28
    for off in range(0, m, step):
        blk = b[off:off + step]
        blk.uniform_(-0.5, 0.5, generator=gen)
        blk.add_(a[off:off + step])
    # a few degenerate and long segments at the boundaries too
    rows = torch.from_numpy(_planted_rows(m, boundaries)[::3]).cuda()
    b[rows] = a[rows]
    return a, b


def seg_call(h, a, b, fn, arg):
    def call(off, c, outs):
        _ok(h, fn(h._h, C.c_void_p(a.data_ptr() + off * 12), C.c_void_p(b.data_ptr() + off * 12), c, 3, L.PC_DEVICE,
                  PC_QUERY_SORTED, arg, _vp(outs[0]), _vp(outs[1])))
    return call


@pytest.mark.parametrize("kind", ["segment", "sweep"])
def test_segments_sorted(cloud, kind):
    """pc_segment_nearest_batch (within 2 m) and pc_sphere_sweep_batch (r = 0.3), PC_QUERY_SORTED, 2^30 + 17 rows: the
    midpoint ordering at >= 2^30 rows."""
    pts, half, ko = cloud
    m = G + 17
    with handle(pts) as h:
        # endpoints, midpoints, outputs, sort buffers and scratch, one sub-batch's outputs
        _budget(m * 24 + m * 16 + m * 8 + m * 16 + m * 2 + SUB * 8, f"{kind}, {m} rows")
        a, b = make_segments(m, half, pts, [G], seed=13 if kind == "segment" else 15)
        idx = torch.empty(m, dtype=torch.int32, device="cuda")
        f = torch.empty(m, dtype=torch.float32, device="cuda")
        fn, arg = (h._L.pc_segment_nearest_batch, SEG_RANGE) if kind == "segment" else (h._L.pc_sphere_sweep_batch, SWEEP_R)
        call = seg_call(h, a, b, fn, arg)
        call(0, m, [idx, f])
        check_sub_batches(call, m, 1, [idx, f], what=kind)
        rows = sample_rows(m, [G], 14, 20_000)
        sa, sb, gi, gf = take(a, rows), take(b, rows), take(idx, rows), take(f, rows)
        if kind == "segment":
            bi, bf = brute_segment(pts, sa, sb, SEG_RANGE)
            want = bf.astype(np.float32)
        else:
            bi, bf = brute_sweep(pts, sa, sb, SWEEP_R)
            want = round_down_f32(bf)
        fin = np.isfinite(sa).all(1) & np.isfinite(sb).all(1)
        bad = np.nonzero((gi != bi) | ((gf.view(np.uint32) != want.view(np.uint32)) & fin))[0]
        assert bad.size == 0, f"{bad.size} rows differ, first {rows[bad[:4]].tolist()}: {gi[bad[:4]]} {gf[bad[:4]]} vs {bi[bad[:4]]} {want[bad[:4]]}"
        assert np.isnan(gf[~fin]).all() and (~fin).sum() > 0
        assert (gi >= 0).sum() > 1000, "too few segments near the cloud"


# ---- range ----------------------------------------------------------------------------------------------------------------
RANGE_R = 0.65               # about 110 hits per row on the forest's surfaces
RANGE_LONG = 2.5             # every 1021st row: about 1600 hits, past what the counting pass captures (512)


def range_radii(m):
    r = torch.full((m,), RANGE_R, dtype=torch.float64, device="cuda")
    r[::1021] = RANGE_LONG
    return r


def range_queries(m, pts, seed):
    """Queries on the cloud's surfaces: cloud points + 0.1 m noise."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    tp = torch.from_numpy(pts).cuda()
    q = torch.empty((m, 3), dtype=torch.float32, device="cuda")
    step = 1 << 24
    for off in range(0, m, step):
        c = min(step, m - off)
        pick = torch.randint(0, len(pts), (c,), generator=gen, device="cuda")
        q[off:off + c] = tp[pick] + 0.1 * torch.randn((c, 3), generator=gen, device="cuda")
    return q


def range_call(h, q, rr, kind, max_nn):
    def call(off, c, off_t, idx_t, d2_t, cap):
        qp, rp = C.c_void_p(q.data_ptr() + off * 12), C.c_void_p(rr.data_ptr() + off * 8)
        ip = _vp(idx_t) if idx_t is not None else C.c_void_p(0)
        if kind == "range":
            return h._L.pc_range_batch(h._h, qp, c, 3, L.PC_DEVICE, rp, 0, _vp(off_t), ip, cap)
        dp = _vp(d2_t) if d2_t is not None else C.c_void_p(0)
        return h._L.pc_range_sorted_batch(h._h, qp, c, 3, L.PC_DEVICE, rp, 0, max_nn, _vp(off_t), ip, dp, cap)
    return call


@pytest.mark.parametrize("kind,max_nn", [("range", 0), ("sorted", 0), ("sorted", 64)],
                         ids=["range", "sorted_all", "sorted_max64"])
def test_range_past_2_31_hits(cloud, kind, max_nn):
    """pc_range_batch / pc_range_sorted_batch, PC_DEVICE: enough rows for more than 2^31 hits in all (int64 offsets, begin + i
    stores, the long-list walks and sorts of every 1021st row); PC_ECAP with complete offsets at cap = 2^31."""
    pts, half, ko = cloud
    with handle(pts) as h:
        # the batch size from the hits of a 2^20-row prefix: 5 % past 2^31 (max_nn = 64: every row cut to at most 64)
        probe = range_queries(1 << 20, pts, seed=17)
        po = torch.zeros((1 << 20) + 1, dtype=torch.int64, device="cuda")
        _ok(h, range_call(h, probe, range_radii(1 << 20), kind, max_nn)(0, 1 << 20, po, None, None, 0))
        mean = int(po[-1]) / (1 << 20)
        m = int(1.05 * (1 << 31) / mean) + 1
        assert m < 1 << 28, f"{mean} hits per row"
        del probe, po
        per_hit = 4 if kind == "range" else 8
        est = int(m * mean * 1.1)
        # queries, offsets, rows, the staging scratch (twice the parked rows) and one sub-batch's rows
        _budget(m * 20 + m * 8 * 4 + est * per_hit * 3 + (est // 8) * per_hit, f"{kind} max_nn={max_nn}, {m} rows")
        q = range_queries(m, pts, seed=19)
        rr = range_radii(m)
        rows_sp = _planted_rows(m, [m // 2])
        sp = _specials(pts, np.random.default_rng(19))
        q[torch.from_numpy(rows_sp).cuda()] = torch.from_numpy(sp[np.arange(len(rows_sp)) % len(sp)]).cuda()
        call = range_call(h, q, rr, kind, max_nn)
        off_t = torch.zeros(m + 1, dtype=torch.int64, device="cuda")
        _ok(h, call(0, m, off_t, None, None, 0))
        total = int(off_t[-1])
        assert total > 1 << 31, f"{total} hits"
        print(f"{kind} max_nn={max_nn}: {m} rows, {total} hits")
        idx = torch.empty(total, dtype=torch.int32, device="cuda")
        d2 = torch.empty(total, dtype=torch.float32, device="cuda") if kind == "sorted" else None
        off2 = torch.full((m + 1,), -5, dtype=torch.int64, device="cuda")
        # a cap below the total: PC_ECAP, and the offsets still complete
        rc = call(0, m, off2, idx, d2, 1 << 31)
        assert rc == L.PC_ECAP
        assert torch.equal(off2, off_t), "PC_ECAP: offsets incomplete"
        _ok(h, call(0, m, off2, idx, d2, total))
        assert torch.equal(off2, off_t)
        # every row against sub-batches of 2^22 rows (< 2^31 hits each)
        sub = 1 << 22
        for s0 in range(0, m, sub):
            c = min(sub, m - s0)
            so = torch.zeros(c + 1, dtype=torch.int64, device="cuda")
            _ok(h, call(s0, c, so, None, None, 0))
            b0, b1 = int(off_t[s0]), int(off_t[s0 + c])
            assert torch.equal(so, off_t[s0:s0 + c + 1] - b0), f"row lengths of the sub-batch at {s0}"
            si = torch.empty(max(b1 - b0, 1), dtype=torch.int32, device="cuda")
            sd = torch.empty(max(b1 - b0, 1), dtype=torch.float32, device="cuda") if d2 is not None else None
            _ok(h, call(s0, c, so, si, sd, b1 - b0))
            assert torch.equal(si[:b1 - b0], idx[b0:b1]), f"indices of the sub-batch at {s0}"
            if d2 is not None:
                assert torch.equal(_bits(sd[:b1 - b0]), _bits(d2[b0:b1])), f"d2 of the sub-batch at {s0}"
        # sampled rows against the brute force; rows around the entries 2^31
        cross = int(torch.searchsorted(off_t, torch.tensor([1 << 31], dtype=torch.int64, device="cuda"), right=True)) - 1
        assert off_t[cross] <= 1 << 31 < off_t[cross + 1]
        rows = sample_rows(m, [cross, m // 2], 20, 4_000)
        qs = take(q, rows)
        bo, bi, bd = brute_range_sorted(pts, qs, take(rr, rows), max_nn)
        go = off_t.cpu().numpy()
        lens = go[rows + 1] - go[rows]
        assert (lens == np.diff(bo)).all(), "row lengths differ from the brute force"
        gi = np.concatenate([idx[go[r]:go[r + 1]].cpu().numpy() for r in rows[lens > 0]]) if (lens > 0).any() else np.zeros(0, np.int32)
        if kind == "range":
            # ascending original index per row
            row_of = np.repeat(np.arange(len(rows)), lens)
            bi = bi[np.lexsort((bi, row_of))]
        else:
            gd = np.concatenate([d2[go[r]:go[r + 1]].cpu().numpy() for r in rows[lens > 0]])
            assert (gd.view(np.uint32) == bd.astype(np.float32).view(np.uint32)).all(), "d2 differs from the brute force"
        assert (gi == bi).all(), "indices differ from the brute force"
        assert lens.sum() > 100_000 and (take(rr, rows) == RANGE_LONG).sum() > 20


# ---- distance field -------------------------------------------------------------------------------------------------------
def test_distance_field_past_2_32_voxels(cloud):
    """pc_distance_field, 2048 x 2048 x 1025 voxels (more than 2^32) within 1 m: one PC_DEVICE launch against the PC_HOST
    layer chunks (the centres of a shifted sub-lattice round differently, so the chunks are the full-field check)."""
    pts, half, ko = cloud
    nx, ny, nz = 2048, 2048, 1025
    n = nx * ny * nz
    assert n > 1 << 32
    voxel = 2 * half / nx
    origin = (-half, -half, -0.5)
    _host_budget(n * 8, f"distance field, {n} voxels")
    with handle(pts) as h:
        _budget(n * 8 + (1 << 31), f"distance field, {n} voxels")
        dist, idx = h.distance_field(origin, voxel, (nx, ny, nz), FIELD_R, on_device=True)
        torch.cuda.synchronize()
        hd, hi = h.distance_field(origin, voxel, (nx, ny, nz), FIELD_R)
        dist, idx, hd, hi = dist.reshape(-1), idx.reshape(-1), hd.reshape(-1), hi.reshape(-1)
        step = 1 << 28
        for off in range(0, n, step):
            c = min(step, n - off)
            a = torch.from_numpy(hi[off:off + c]).cuda()
            b = torch.from_numpy(hd[off:off + c]).cuda()
            if not (torch.equal(a, idx[off:off + c]) and torch.equal(_bits(b), _bits(dist[off:off + c]))):
                bad = torch.nonzero((a != idx[off:off + c]) | (_bits(b) != _bits(dist[off:off + c])))[:4, 0].cpu().numpy() + off
                raise AssertionError(f"voxels {bad.tolist()}: PC_DEVICE differs from PC_HOST")
        rows = sample_rows(n, [1 << 31, 1 << 32], 22, 20_000)
        i, j, k = rows % nx, (rows // nx) % ny, rows // (nx * ny)
        c = np.stack([(o + (v.astype(np.float64) + 0.5) * voxel) for o, v in zip(origin, (i, j, k))], 1).astype(np.float32)
        bi, bd = brute_knn(pts, c, 1, FIELD_R)
        want = np.where(bi[:, 0] >= 0, np.sqrt(bd[:, 0]), np.inf).astype(np.float32)
        gi, gd = hi[rows], hd[rows]
        bad = np.nonzero((gi != bi[:, 0]) | (gd.view(np.uint32) != want.view(np.uint32)))[0]
        assert bad.size == 0, f"{bad.size} voxels differ from the brute force, first {rows[bad[:4]].tolist()}"
        assert (gi >= 0).sum() > 1000
