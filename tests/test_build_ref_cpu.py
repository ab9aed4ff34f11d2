"""Checks of the numpy restatement of the index build (tests/build_ref.py) that tests/test_index_build_gpu.py compares the GPU
build with: its Hilbert keys are a curve, its 10-bit keys are those of the host model, its tree is the tree pc_lbvh_node and
pc_lbvh_children define, and its records hold tight boxes over a partition of the cloud."""
import os
import subprocess

import numpy as np
import pytest

import build_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("build_ref") / "build_ref_check")
    subprocess.run(["g++", "-std=c++14", "-O2", "-o", exe, os.path.join(ROOT, "tests", "c", "build_ref_check.cpp")],
                   check=True, capture_output=True)
    return exe


def _run(exe, mode, arr, out_dtype, tmp_path):
    fi, fo = str(tmp_path / f"{mode}.in"), str(tmp_path / f"{mode}.out")
    np.ascontiguousarray(arr).tofile(fi)
    r = subprocess.run([exe, mode, fi, fo], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr
    return np.fromfile(fo, out_dtype)


@pytest.mark.parametrize("bits", [2, 3, 4, 5, 6, 7])
def test_hilbert_keys_are_a_curve(bits):
    """Every cell of a 2^bits cube gets its own key in [0, 2^(3 bits)), and consecutive keys are face-adjacent cells."""
    s = 1 << bits
    g = np.stack(np.meshgrid(*(np.arange(s, dtype=np.uint32),) * 3, indexing="ij"), -1).reshape(-1, 3)
    k = R.hilbert_keys(g, bits)
    order = np.argsort(k)
    assert (k[order] == np.arange(s ** 3, dtype=np.uint64)).all()
    step = np.abs(np.diff(g[order].astype(np.int64), axis=0)).sum(1)
    assert (step == 1).all()


def test_ten_bit_keys_match_the_host_model(harness, tmp_path):
    rng = np.random.default_rng(0)
    c = rng.integers(0, 1024, size=(200_000, 3), dtype=np.uint32)
    c[:8] = [[0, 0, 0], [1023, 1023, 1023], [1023, 0, 0], [0, 1023, 0], [0, 0, 1023], [512, 511, 512], [1, 2, 3], [1023, 1022, 1]]
    want = _run(harness, "keys", c, np.uint32, tmp_path)
    assert (R.hilbert_keys(c, 10) == want.astype(np.uint64)).all()


def _clouds():
    rng = np.random.default_rng(1)
    out = {}
    for n in (5, 6, 8, 9, 16, 17, 33, 100, 257, 1000, 4097):
        out[f"normal{n}"] = rng.normal(size=(n, 3)).astype(np.float32)
    out["all_equal"] = np.tile(np.float32([[1.5, -2.0, 0.75]]), (300, 1))
    lat = rng.integers(0, 3, size=(2000, 3)).astype(np.float32)               # 27 cells: long runs of equal keys
    out["duplicates"] = lat
    runs = np.repeat(rng.normal(size=(40, 3)).astype(np.float32), rng.integers(1, 30, 40), axis=0)
    out["runs"] = runs[rng.permutation(len(runs))]
    out["collinear"] = np.column_stack([np.linspace(0, 1, 777), np.zeros(777), np.zeros(777)]).astype(np.float32)
    return out


CLOUDS = _clouds()


@pytest.mark.parametrize("name", sorted(CLOUDS))
def test_tree_topology_matches_the_node_function(harness, tmp_path, name):
    """Top-down splits (tests/build_ref.py) and Karras' per-node ranges (lbvh.cuh, built for the host) are two constructions of
    one tree: the same node ids carry the same range, split and children, and exactly the nodes of more than PC_LEAF points
    are reachable from the root."""
    ref = R.BuildRef(CLOUDS[name])
    n = ref.n
    got = _run(harness, "nodes", ref.keys.astype(np.uint64), np.int64, tmp_path).reshape(n - 1, 7)
    size = got[:, 1] - got[:, 0] + 1
    assert ((size > R.PC_LEAF) == ref.reachable).all()
    m = ref.reachable
    assert (got[m, 0] == ref.first[m]).all() and (got[m, 1] == ref.last[m]).all() and (got[m, 2] == ref.split[m]).all()
    words = ref.records[m][:, [6, 14, 7, 15]].astype(np.int64)
    assert (got[m, 3:] == words).all()


@pytest.mark.parametrize("name", sorted(CLOUDS))
def test_records_partition_the_cloud_with_tight_boxes(name):
    p = CLOUDS[name]
    ref = R.BuildRef(p)
    n = ref.n
    assert (np.sort(ref.points[:n, 3]) == np.arange(n)).all()
    assert (ref.points[n:] == ref.points[n - 1]).all()
    assert (ref.points[:n, :3].view(np.float32) == p[ref.order]).all()
    sp = ref.points[:n, :3].view(np.float32)
    rec = ref.records.view(np.float32)
    covered = np.zeros(n, np.int64)
    for i in np.flatnonzero(ref.reachable):
        f, l, s = ref.first[i], ref.last[i], ref.split[i]
        for c, (cf, cl) in enumerate(((f, s), (s + 1, l))):
            r, k = int(ref.records[i, 6 + c]), int(ref.records[i, 14 + c])
            assert k == cl - cf + 1
            if r & R.PC_REF_LEAF:
                assert k <= R.PC_LEAF and r & 0x7fffffff == cf
                covered[cf:cl + 1] += 1
            else:
                assert k > R.PC_LEAF and r == (s if c == 0 else s + 1)
                assert ref.first[r] == cf and ref.last[r] == cl and ref.depth[r] == ref.depth[i] + 1
            lo = [rec[i, 2 * a + c] for a in range(3)]
            hi = [rec[i, 8 + 2 * a + c] for a in range(3)]
            assert (np.array(lo) == sp[cf:cl + 1].min(0)).all() and (np.array(hi) == sp[cf:cl + 1].max(0)).all()
    assert (covered == 1).all()            # the leaves partition the cloud
    assert ref.first[0] == 0 and ref.last[0] == n - 1


def test_frame_ignores_points_with_a_non_finite_coordinate():
    p = np.random.default_rng(2).normal(size=(1000, 3)).astype(np.float32)
    q = p.copy()
    q[[3, 50, 700]] = [[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf]]
    lo, hi, inv = R.frame(q)
    keep = np.ones(1000, bool)
    keep[[3, 50, 700]] = False
    lo2, hi2, inv2 = R.frame(p[keep])
    assert (lo == lo2).all() and (hi == hi2).all() and inv == inv2 and inv > 0
    lo, hi, inv = R.frame(np.full((7, 3), np.nan, np.float32))
    assert (lo == np.inf).all() and (hi == -np.inf).all() and inv == 0
    ref = R.BuildRef(np.full((7, 3), np.nan, np.float32))
    assert (ref.keys == 0).all() and (ref.order == np.arange(7)).all()


def test_cells_on_boundaries_and_at_hi():
    """A point at hi lands in the last cell, not past it (the 1 - 1e-6 factor), and cell boundaries truncate downwards."""
    bits = 10
    p = np.array([[0, 0, 0], [1, 1, 1], [0.5, 0.25, 0.125]], np.float32)
    lo, hi, inv = R.frame(p)
    c = R.cells(p, lo, inv, bits)
    assert (c[0] == 0).all() and (c[1] == 1023).all()
    assert (c[2] == [511, 255, 127]).all()          # 2^bits (1 - 1e-6) * 0.5 = 511.9995 -> 511
    assert inv == np.float32(np.float32(1024) * np.float32(np.float32(1) - np.float32(1e-6)))
