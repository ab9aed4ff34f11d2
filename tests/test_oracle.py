"""CPU tests: the oracle restatement against (a) golden vectors produced by the unmodified reference
kd-tree and (b) the reference library itself when oracle/_ref is present."""
import numpy as np
import pytest

import oracle
from pointcloudtraj_b200 import synth

CASES = ["forest_lattice", "forest_jitter", "uniform"]


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_golden_nearest(golden_dir, name):
    g = np.load(f"{golden_dir}/{name}.npz")
    ko = oracle.KdOracle().build(g["pts"], g["order"])
    idx, d2 = ko.nearest(g["q"])
    assert (idx == g["nn_idx"]).all()          # including the reference's choice among tied points
    assert (d2 == g["nn_d2"]).all()            # bitwise fp64


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_golden_range(golden_dir, name):
    g = np.load(f"{golden_dir}/{name}.npz")
    ko = oracle.KdOracle().build(g["pts"], g["order"])
    off, lst = ko.range(g["range_q"], float(g["range_r"]))
    assert (off == g["range_off"]).all()
    assert (lst == g["range_idx"]).all()       # same iteration order as the reference's result set


def test_known_answers(golden_dir):
    k = np.load(f"{golden_dir}/kat.npz")
    z = np.zeros((1, 3), np.float32)
    two = np.array([[1, 0, 0], [-1, 0, 0]], np.float32)
    assert oracle.KdOracle().build(two).nearest(z)[0].tolist() == k["tie_two_first_inserted_wins"].tolist() == [0]
    assert oracle.KdOracle().build(two, [1, 0]).nearest(z)[0].tolist() == k["tie_two_reversed_insert"].tolist() == [1]
    dup = np.array([[2, 2, 2]] * 3, np.float32)
    assert oracle.KdOracle().build(dup).nearest(np.array([[2.5, 2, 2]], np.float32))[0].tolist() == k["three_duplicates"].tolist()
    bp = np.array([[0.5, 5, 5], [0.5, 0, 0]], np.float32)
    ko = oracle.KdOracle().build(bp)
    # range boundary asymmetry of the reference (kdtree.c:273 inclusive vs :283 strict)
    assert ko.range(np.array([[-0.5, 0, 0]], np.float32), 1.0)[0].tolist() == k["range_boundary_left"].tolist() == [0, 0]
    assert ko.range(np.array([[1.5, 0, 0]], np.float32), 1.0)[0].tolist() == k["range_boundary_right"].tolist() == [0, 1]
    empty = oracle.KdOracle().build(np.zeros((0, 3), np.float32))
    i, d = empty.nearest(np.zeros((2, 3), np.float32))
    assert i.tolist() == k["empty_idx"].tolist() == [-1, -1] and np.isinf(d).all()
    assert empty.range(np.zeros((2, 3), np.float32), 1.0)[0].tolist() == [0, 0, 0]


@pytest.mark.skipif(not oracle.have_reference(), reason="needs the upstream pointcloudTraj kd-tree compiled into oracle/_ref (make -C oracle REF=<pointcloudTraj checkout>)")
@pytest.mark.parametrize("variant,n,m,lat", [("L", 30000, 6000, 0.5), ("J", 30000, 6000, 0.0)])
def test_oracle_equals_reference_library(variant, n, m, lat):
    pts, half = synth.forest_cloud(n, seed=4, variant=variant, return_half=True)
    q = synth.rrt_queries(m, half, seed=5, lattice_frac=lat)
    order = np.random.default_rng(7).permutation(n)
    ko = oracle.KdOracle().build(pts, order)
    kr = oracle.KdReference().build(pts, order)
    i1, d1 = ko.nearest(q)
    i2, d2 = kr.nearest(q)
    assert (i1 == i2).all() and (d1 == d2).all()
    o1, l1 = ko.range(q[:500], 0.9)
    o2, l2 = kr.range(q[:500], 0.9)
    assert (o1 == o2).all() and (l1 == l2).all()
    # exactness: the tree search returns the brute-force fp64 minimum distance
    _, db, _ = oracle.brute_nearest(pts, q[:1000])
    assert (d1[:1000] == db).all()


@pytest.mark.skipif(not oracle.have_reference(), reason="needs the upstream pointcloudTraj kd-tree compiled into oracle/_ref (make -C oracle REF=<pointcloudTraj checkout>)")
def test_radius_restatement_matches_reference_harness():
    pts, half = synth.forest_cloud(20000, seed=2, variant="J", return_half=True)
    q = synth.rrt_queries(4000, half * 1.5, seed=3)
    order = np.random.default_rng(1).permutation(len(pts))
    P = oracle.RadiusParams.make(0.25, 1.5, 12.0, (1.0, -2.0, 2.0))
    r1, _ = oracle.KdOracle().build(pts, order).radius_batch(P, q)
    r2 = oracle.KdReference().build(pts, order).radius_batch(P, q)
    assert (r1 == r2).all()
    assert (r1 == P.max_radius - P.search_margin).any()      # early-outs exercised
    assert (r1 == P.max_radius).any() and (r1 < 0).any()     # clamp and collision exercised


def test_radius_search_semantics():
    # corridor_finder.cpp:113-133 on a single obstacle point
    ko = oracle.KdOracle().build(np.array([[0, 0, 0]], np.float32))
    P = oracle.RadiusParams.make(0.25, 1.5, 30.0, (0.0, 0.0, 0.0))
    assert ko.radius_search(P, [1.0, 0, 0])[0] == 1.0 - 0.25
    assert ko.radius_search(P, [5.0, 0, 0])[0] == 1.5                     # clamp to max_radius
    assert ko.radius_search(P, [0.1, 0, 0])[0] < 0                        # collision
    assert ko.radius_search(P, [40.0, 0, 0])[0] == 1.5 - 0.25             # outside sample_range + max_radius
    empty = oracle.KdOracle().build(np.zeros((0, 3), np.float32))
    assert empty.radius_search(P, [1.0, 0, 0])[0] == 1.5 - 0.25           # empty cloud


def test_bezier_restatement():
    # Bernstein basis sums to one; end points are interpolated; binomials as bezier_base.cpp:35-48
    assert [oracle.binomial(6, k) for k in range(7)] == [1, 6, 15, 20, 15, 6, 1]
    assert oracle.binomial(12, 6) == 924
    rng = np.random.default_rng(0)
    for n in (4, 6, 8, 12):
        c = rng.normal(size=3 * (n + 1))
        assert np.allclose(oracle.bezier_pos(c, n, 0.0), c[[0, n + 1, 2 * n + 2]])
        assert np.allclose(oracle.bezier_pos(c, n, 1.0), c[[n, 2 * n + 1, 3 * n + 2]])
        assert np.allclose(oracle.bezier_pos(np.ones(3 * (n + 1)), n, 0.37), 1.0)


def test_check_safe_trajectory_walk():
    # one straight segment flying into a wall point: p(t) = T * B(u); control points are stored scaled by 1/T
    ko = oracle.KdOracle().build(np.array([[5.0, 0, 1.0]], np.float32))
    P = oracle.RadiusParams.make(0.25, 1.5, 30.0, (0.0, 0.0, 1.0))
    T = 4.0
    n = 4
    xs = np.linspace(0, 8, n + 1) / T
    coef = np.concatenate([xs, np.zeros(n + 1), np.full(n + 1, 1.0 / T)])[None, :]
    out = ko.check_safe_trajectory(P, [n], [T], coef, t_now=0.0, stop_time=10.0)
    # samples at t = 0, 0.02, ... < 4.0 -> 200 samples (t_accu never exceeds 10)
    assert out["n_samples"] == 200
    x = out["pts"][:, 0]
    assert np.allclose(x, np.arange(200) * 0.02 * 2.0, atol=1e-5)
    first = int(np.nonzero(np.abs(x.astype(np.float64) - 5.0) < 0.25)[0][0])
    assert out["first_hit"] == first
    assert out["min_radius"] < 0
    # horizon: only samples with accumulated time <= stop_time
    out2 = ko.check_safe_trajectory(P, [n], [T], coef, t_now=0.0, stop_time=1.0)
    assert out2["n_samples"] in (49, 50) and out2["first_hit"] == -1
