"""Parity at the sizes BASELINE.json's configs name (the other GPU tests use smaller clouds so that the oracle stays fast):
C2 radius batches on the 1M-point bench map with both parameter sets, a C3 LiDAR stream of 20 frames of 300k points with
per-frame parity, the C4 clearance batch (5M points, 10^4 trajectories x 10^3 samples; oracle on a subsample of the
trajectories), and -- opt-in, PC_RUN_C5=1 -- a spot check on the 100M-point cloud of C5."""
import os

import numpy as np
import pytest

import oracle
from pointcloudtraj_b200 import PC_RADIUS_FULL_NN, PcRadiusParams, PointCloudIndex, synth

pytestmark = pytest.mark.gpu

CLEAN_DEMO = dict(search_margin=0.25, max_radius=1.5, sample_range=30.0)      # clean_demo.launch:31-34
SIMULATION = dict(search_margin=0.0, max_radius=5.0, sample_range=30.0)       # simulation.launch:24-27


def _cpu_tree(pts, seed=0):
    """The unmodified reference kd-tree when oracle/_ref holds it, else the oracle's C restatement (kd_oracle.c).  The
    restatement is not the original: test_oracle.py pins it to the reference's stored answers in tests/golden."""
    order = np.random.default_rng(seed).permutation(len(pts))
    if oracle.have_reference():
        return oracle.KdReference().build(pts, order), True
    return oracle.KdOracle().build(pts, order), False


def _cpu_radius(tree, is_ref, params, start, q):
    P = oracle.RadiusParams.make(start=start, **params)
    return tree.radius_batch(P, q) if is_ref else tree.radius_batch(P, q)[0]


def test_c2_radius_parity_on_the_1m_point_map():
    """The bench workload itself: 1M-point map, both parameter sets, bounded and full-NN, against the CPU kd-tree of
    _cpu_tree (the reference's own when oracle/_ref is present, else the oracle's restatement)."""
    pts, half = synth.forest_cloud(1_000_000, seed=1, variant="J", return_half=True)
    q = synth.rrt_queries(250_000, half, seed=21)
    tree, is_ref = _cpu_tree(pts)
    start = (0.0, 0.0, 2.0)
    with PointCloudIndex(max_points=len(pts)) as ix:
        ix.build(pts)
        for params in (CLEAN_DEMO, SIMULATION):
            ref = _cpu_radius(tree, is_ref, params, start, q).astype(np.float32)
            P = PcRadiusParams.make(start=start, **params)
            r, idx = ix.radius(q, P, want_idx=True)
            assert (r == ref).all()
            r_full, idx_full = ix.radius(q, P, flags=PC_RADIUS_FULL_NN, want_idx=True)
            assert (r_full == ref).all()
            found = idx >= 0
            assert (idx[found] == idx_full[found]).all() and found.any() and (~found).any()
        ridx, rd2 = tree.nearest(q[:100_000])
        gi, gd = ix.nearest(q[:100_000])
        assert (gi == ridx).all() and (gd == rd2.astype(np.float32)).all()


def test_c3_lidar_stream_20_frames_of_300k_points():
    """10 Hz LiDAR stream: every frame is the 300k map points nearest to a sensor that moves 0.3 m per frame (gathered with
    pc_sphere_gather, checked against numpy), followed by a full index rebuild and 1M radius queries; per-frame parity of a
    query subsample against a kd-tree built on that frame."""
    N, M, FRAMES = 300_000, 1_000_000, 20
    world, half = synth.forest_cloud(2_000_000, seed=3, variant="J", return_half=True)
    rng = np.random.default_rng(4)
    build_ms = []
    with PointCloudIndex(max_points=len(world)) as ix_map, PointCloudIndex(max_points=N) as ix:
        ix_map.build(world)
        for k in range(FRAMES):
            sensor = np.array([-10.0 + 0.3 * k, -10.0 + 0.3 * k, 2.0])
            seen = ix_map.sphere_gather(sensor, 25.0)
            d2 = ((world[seen].astype(np.float64) - sensor.astype(np.float32).astype(np.float64)) ** 2).sum(1)
            if k % 5 == 0:                                                  # the gather itself against numpy
                all_d2 = ((world.astype(np.float64) - sensor.astype(np.float32).astype(np.float64)) ** 2)
                brute = np.nonzero((all_d2[:, 0] + all_d2[:, 1]) + all_d2[:, 2] <= 625.0)[0]
                assert (seen == brute).all()
            assert len(seen) >= N
            frame = np.ascontiguousarray(world[seen[np.argsort(d2, kind="stable")[:N]]])
            ix.build(frame)
            build_ms.append(ix.last_build_ms())
            q = (sensor + rng.uniform([-25, -25, -1.4], [25, 25, 2.0], size=(M, 3))).astype(np.float32)
            P = PcRadiusParams.make(start=tuple(sensor), **CLEAN_DEMO)
            r = ix.radius(q, P)
            sub = rng.choice(M, 15_000, replace=False)
            tree, is_ref = _cpu_tree(frame, seed=k)
            ref = _cpu_radius(tree, is_ref, CLEAN_DEMO, tuple(sensor), q[sub]).astype(np.float32)
            assert (r[sub] == ref).all(), f"frame {k}"
    assert np.median(build_ms) < 1.0                                        # the north star's rebuild budget per 300k-point frame


def test_c4_clearance_batch_at_full_size():
    """10^4 piecewise trajectories x up to 10^3 samples against the 5M-point cloud in ONE pc_clearance_batch call; the oracle
    (restated checkSafeTrajectory, pinned to the compiled reference by test_planner_ref.py) on a subsample of 200."""
    pts, half = synth.forest_cloud(5_000_000, seed=2, variant="J", return_half=True)
    n_traj = 10_000
    tr = synth.bezier_trajectories(n_traj, half * 0.9, seed=4)
    first, order, T, off, coef = tr["traj_first_seg"], tr["seg_order"], tr["seg_T"], tr["seg_coef_off"], tr["coef"]
    start = (0.0, 0.0, 2.0)
    params = dict(search_margin=0.25, max_radius=1.5, sample_range=60.0)
    with PointCloudIndex(max_points=len(pts)) as ix:
        ix.build(pts)
        fh, mr, ns = ix.clearance(first, order, T, off, coef, PcRadiusParams.make(start=start, **params), dt=0.02, horizon=20.0)
    assert ns.max() >= 990 and ns.sum() > 3_000_000 and (fh >= 0).any() and (fh < 0).any()
    ko = oracle.KdOracle().build(pts, np.random.default_rng(1).permutation(len(pts)))
    P = oracle.RadiusParams.make(start=start, **params)
    for t in np.random.default_rng(2).choice(n_traj, 200, replace=False):
        segs = list(range(first[t], first[t + 1]))
        mat = np.zeros((len(segs), 3 * (int(order[segs].max()) + 1)))
        for r_, s in enumerate(segs):
            c = coef[off[s]:off[s + 1]]
            mat[r_, : len(c)] = c
        ref = ko.check_safe_trajectory(P, order[segs], T[segs], mat, t_now=0.0, stop_time=20.0, cap=2048)
        assert ns[t] == ref["n_samples"] and fh[t] == ref["first_hit"]
        assert mr[t] == np.float32(ref["min_radius"])


@pytest.mark.skipif(os.environ.get("PC_RUN_C5") != "1", reason="opt-in (PC_RUN_C5=1): 100M points, ~2 min of host-side generation")
def test_c5_spot_check_on_100m_points():
    """C5: 100M-point cloud (a 25M-point forest and three shifted copies of it, 63-bit keys), 10^7 unbounded nearest queries;
    spot check of 300 queries against an fp64 brute force."""
    base, half = synth.forest_cloud(25_000_000, seed=5, variant="J", return_half=True)
    shifts = np.array([[0, 0, 0], [2 * half + 3, 0, 0], [0, 2 * half + 3, 0], [2 * half + 3, 2 * half + 3, 0]], np.float32)
    pts = np.concatenate([base + s for s in shifts])
    del base
    q = synth.rrt_queries(10_000_000, half, seed=6) + shifts[np.random.default_rng(7).integers(0, 4, 10_000_000)]
    with PointCloudIndex(max_points=len(pts)) as ix:
        ix.build(pts)
        idx, d2 = ix.nearest(q)
        bi, bd, _ = oracle.brute_nearest(pts, q[:300])
        assert (idx[:300] == bi).all() and (d2[:300] == bd.astype(np.float32)).all()
        sel = np.random.default_rng(8).permutation(len(pts))[:1_000_000]
        i2, e2 = ix.nearest(pts[sel])
        assert (e2 == 0).all() and (i2 == sel).all()
