"""The built index, record for record, against the numpy restatement of the build (tests/build_ref.py).

Query answers cannot see a box looser than tight, a badly split leaf, an unstable sort or wrong walk seeds: all of them keep
every answer exact and only make traversals slower.  So these tests read the device arrays behind pc_index_view (records,
points and the 100 seed words behind the points) and compare them with the reference:
  * header: n_points, n_nodes, root, root_count exactly, bbox with ==;
  * points: bitwise, the PC_LEAF pad copies included;
  * records of the nodes reachable from the root: child references and counts bitwise, box words by value (+0 == -0);
    records of collapsed nodes are documented as unwritten and not compared;
  * seeds: the counts, then the multisets of inner references and of (reference, count) leaf pairs.
The cases pin the build's path switches (ITEMS 8 -> 16 above 2^21 points, 30- -> 63-bit keys above 4 Mi, the three-kernel
sort of PC_ONESWEEP=0), its call paths (stride 3 / 4, PC_HOST / PC_DEVICE, handles that grow and shrink) and clouds that are
hard on a build (equal keys, degenerate extents, far offsets, cell boundaries, non-finite coordinates)."""
import os

import numpy as np
import pytest

import build_ref as R
from pointcloudtraj_b200 import PointCloudIndex, synth

pytestmark = pytest.mark.gpu

MI4 = 1 << 22
BOX_WORDS = [0, 1, 2, 3, 4, 5, 8, 9, 10, 11, 12, 13]
LINK_WORDS = [6, 7, 14, 15]


class _DeviceWords:
    """int32 words of device memory, for torch.as_tensor (the index's arrays are read after pc_index_sync)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (int(ptr), False), "version": 2}


def snapshot(ix):
    import torch
    ix.sync()
    v = ix.view()
    n, m = int(v.n_points), int(v.n_nodes)
    words = 16 * m + 4 * (n + R.PC_LEAF) + R.SEED_WORDS
    a = torch.as_tensor(_DeviceWords(v.records, words), device=f"cuda:{ix.device}").cpu().numpy().view(np.uint32)
    return dict(n=n, n_nodes=m, root=int(v.root), root_count=int(v.root_count),
                lo=np.array(v.bbox_lo[:], np.float32), hi=np.array(v.bbox_hi[:], np.float32),
                rec=a[:16 * m].reshape(m, 16), pts=a[16 * m:16 * m + 4 * (n + R.PC_LEAF)].reshape(-1, 4),
                seeds=a[16 * m + 4 * (n + R.PC_LEAF):])


def _node_msg(ref, i, what, got, want):
    return (f"{what}: first differing node {i} (points [{ref.first[i]}, {ref.last[i]}], split {ref.split[i]}, depth "
            f"{ref.depth[i]}): got {got}, want {want}")


def check(s, ref, label=""):
    """Assert that snapshot s is the build the reference describes; the message names the first difference."""
    hdr = (s["n"], s["n_nodes"], s["root"], s["root_count"])
    assert hdr == (ref.n, ref.n_nodes, ref.root, ref.root_count), f"{label} header {hdr}"
    assert (s["lo"] == ref.lo).all() and (s["hi"] == ref.hi).all(), f"{label} bbox {s['lo']} {s['hi']} want {ref.lo} {ref.hi}"
    bad = np.flatnonzero((s["pts"] != ref.points).any(1))
    if len(bad):
        k = bad[0]
        raise AssertionError(f"{label} points: {len(bad)} curve positions differ, first {k}: got {s['pts'][k]} "
                             f"(index {s['pts'][k, 3]}), want {ref.points[k]} (index {ref.points[k, 3]})")
    m = np.flatnonzero(ref.reachable)
    got, want = s["rec"][m], ref.records[m]
    bad = np.flatnonzero((got[:, LINK_WORDS] != want[:, LINK_WORDS]).any(1))
    if len(bad):
        i = m[bad[0]]
        raise AssertionError(label + " " + _node_msg(ref, i, "references / counts", s["rec"][i, LINK_WORDS], ref.records[i, LINK_WORDS]))
    gb, wb = got[:, BOX_WORDS].view(np.float32), want[:, BOX_WORDS].view(np.float32)
    bad = np.flatnonzero((gb != wb).any(1))
    if len(bad):
        i = m[bad[0]]
        raise AssertionError(label + " " + _node_msg(ref, i, "boxes [lo0 lo1 x y z | hi0 hi1 x y z]", gb[bad[0]], wb[bad[0]]))
    g, w = s["seeds"], ref.seeds
    assert (g[:2] == w[:2]).all(), f"{label} seed counts {g[:2]} want {w[:2]}"
    ni, nl = int(w[0]), int(w[1])
    sl = slice(R.SEED_INNER, R.SEED_INNER + ni)
    assert (np.sort(g[sl]) == np.sort(w[sl])).all(), f"{label} inner seeds {g[sl]} want {w[sl]}"
    lp = slice(R.SEED_LEAF, R.SEED_LEAF + 2 * nl)
    gp, wp = g[lp].reshape(-1, 2), w[lp].reshape(-1, 2)
    assert (gp[np.lexsort(gp.T[::-1])] == wp[np.lexsort(wp.T[::-1])]).all(), f"{label} leaf seeds {gp} want {wp}"


def written_bytes(s, ref):
    """everything a build writes: the reachable records, the points with their pads, the seed words in use"""
    return (s["rec"][ref.reachable].tobytes(), s["pts"].tobytes(), s["seeds"][ref.seed_mask].tobytes())


# ---- clouds and references, shared by the cases ---------------------------------------------------------------------------
_big = {}


def big_cloud():
    if "p" not in _big:
        _big["p"] = synth.forest_cloud(MI4 + 1, seed=3, variant="J")
    return _big["p"]


_refs = {}


def ref_of(key, p):
    if key not in _refs:
        _refs[key] = R.BuildRef(p)
    return _refs[key]


@pytest.fixture(scope="module")
def ix():
    h = PointCloudIndex(max_points=MI4 + 1, device=0)
    yield h
    h.close()


def _onesweep_off_handle(max_points):
    os.environ["PC_ONESWEEP"] = "0"
    try:
        return PointCloudIndex(max_points=max_points, device=0)
    finally:
        del os.environ["PC_ONESWEEP"]


# ---- sizes: leaf boundaries, CTA boundaries of the fit, ITEMS 8 -> 16, 30- -> 63-bit keys ----------------------------------
SIZES = list(range(1, 10)) + [16, 17, 255, 256, 257, 258, 511, 512, 513, 2047, 2048, 2049, 4095, 4096, 4097, 65537,
                              1 << 21, (1 << 21) + 1, MI4, MI4 + 1]


@pytest.mark.parametrize("n", SIZES)
def test_sizes(ix, n):
    p = big_cloud()[:n]
    ix.build(p)
    check(snapshot(ix), ref_of(("big", n), p), f"n={n}")


# ---- cloud shapes -----------------------------------------------------------------------------------------------------------
def _shape(name):
    rng = np.random.default_rng(11)
    if name == "forest_J":
        return synth.forest_cloud(200_000, seed=5, variant="J")
    if name == "forest_L":
        return synth.forest_cloud(200_000, seed=5, variant="L")
    if name == "uniform":
        return synth.uniform_cloud(300_000, seed=4)
    if name == "identical":
        return np.tile(np.float32([[3.25, -1.5, 0.5]]), (5000, 1))
    if name == "collinear":
        t = rng.uniform(-20, 20, 100_000)
        return (np.outer(t, [0.6, -0.3, 0.2]) + [1.0, 2.0, 3.0]).astype(np.float32)
    if name == "planar":
        return np.column_stack([rng.uniform(-15, 15, 100_000), rng.uniform(-15, 15, 100_000), np.full(100_000, 1.25)]).astype(np.float32)
    if name == "two_clusters":
        a = rng.normal(size=(50_000, 3))
        b = rng.normal(size=(50_000, 3)) + [1e4, 0, 0]
        return np.concatenate([a, b]).astype(np.float32)[rng.permutation(100_000)]
    if name == "offset_1e6":
        return synth.forest_cloud(100_000, seed=8, variant="J") + np.float32(1e6)
    if name == "cell_boundaries":
        # extent 1024 on every axis: integer coordinates are (almost) cell boundaries; hi on every axis, alone and together
        c = rng.integers(0, 1025, size=(60_000, 3)).astype(np.float32)
        c[:8] = [[0, 0, 0], [1024, 1024, 1024], [1024, 0, 0], [0, 1024, 0], [0, 0, 1024], [1024, 1024, 0], [512, 512, 512], [1023, 1023, 1023]]
        c[8:4000, rng.integers(0, 3)] = 1024
        # coordinates whose cell position (v - lo) * inv is an integer after its one rounding, and their neighbours
        inv = R.frame(c)[2]
        k = rng.integers(1, 1024, size=(6000, 3)).astype(np.float32)
        b = k / inv
        c[4000:10000] = b
        c[10000:16000] = np.nextafter(b, np.float32(-np.inf))
        c[16000:22000] = np.nextafter(b, np.float32(np.inf))
        return c
    if name == "no_finite_point":
        p = np.full((3000, 3), np.nan, np.float32)
        p[::3, 0] = np.inf
        p[1::3, 1] = -np.inf
        return p
    raise KeyError(name)


SHAPES = ["forest_J", "forest_L", "uniform", "identical", "collinear", "planar", "two_clusters", "offset_1e6",
          "cell_boundaries", "no_finite_point"]


@pytest.mark.parametrize("name", SHAPES)
def test_cloud_shapes(ix, name):
    p = _shape(name)
    ix.build(p)
    check(snapshot(ix), ref_of(name, p), name)


# ---- call paths -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("space", ["host", "device"])
@pytest.mark.parametrize("stride", [3, 4])
def test_strides_and_memory_spaces(ix, space, stride):
    import torch
    p = _shape("forest_J")
    a = p if stride == 3 else np.column_stack([p, np.full(len(p), np.nan, np.float32)])
    if space == "device":
        a = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    ix.build(a)
    check(snapshot(ix), ref_of("forest_J", p), f"{space} stride {stride}")


@pytest.mark.parametrize("n", [4095, 4096, 4097, MI4 + 1])
def test_three_kernel_sort(n):
    p = big_cloud()[:n]
    h = _onesweep_off_handle(n)
    try:
        h.build(p)
        check(snapshot(h), ref_of(("big", n), p), f"PC_ONESWEEP=0 n={n}")
    finally:
        h.close()


def test_handle_that_grows_shrinks_and_grows():
    h = PointCloudIndex(max_points=0, device=0)
    try:
        for n in ((1 << 21) + 1, 4097, MI4 + 1):
            p = big_cloud()[:n]
            h.build(p)
            check(snapshot(h), ref_of(("big", n), p), f"max_points=0 n={n}")
    finally:
        h.close()


# ---- determinism ------------------------------------------------------------------------------------------------------------
def test_builds_are_deterministic(ix):
    p = _shape("forest_L")
    ref = ref_of("forest_L", p)
    ix.build(p)
    a = written_bytes(snapshot(ix), ref)
    ix.build(p)
    assert written_bytes(snapshot(ix), ref) == a
    ix.build(_shape("uniform"))                 # a different cloud first, then the same one again
    ix.build(p)
    b = written_bytes(snapshot(ix), ref)
    h = PointCloudIndex(max_points=0, device=0)
    try:
        h.build(p)
        assert written_bytes(snapshot(h), ref) == a == b
    finally:
        h.close()


# ---- non-finite coordinates -------------------------------------------------------------------------------------------------
def test_non_finite_points_keep_the_frame_of_the_finite_ones(ix):
    """NaN, +inf and -inf coordinates in a 200 k forest: the frame and the curve order of the finite points are those of the
    build of the finite points alone.  (An infinite coordinate in the frame would give every point key 0.)"""
    p = _shape("forest_J").copy()
    rng = np.random.default_rng(3)
    rows = rng.choice(len(p), 600, replace=False)
    vals = np.float32([np.nan, np.inf, -np.inf])
    for k, r in enumerate(rows):
        p[r, k % 3] = vals[(k // 3) % 3]
    p[rows[:30]] = vals[np.arange(30) % 3][:, None]          # all three coordinates non-finite
    fin = np.isfinite(p).all(1)
    ix.build(p)
    s = snapshot(ix)
    check(s, ref_of("forest_J_nonfinite", p), "non-finite")
    new_id = np.cumsum(fin) - 1
    order_fin = s["pts"][:len(p), 3].astype(np.int64)
    order_fin = new_id[order_fin[fin[order_fin]]]
    ix.build(p[fin])
    t = snapshot(ix)
    assert (s["lo"] == t["lo"]).all() and (s["hi"] == t["hi"]).all()
    assert (order_fin == t["pts"][:int(fin.sum()), 3].astype(np.int64)).all()
