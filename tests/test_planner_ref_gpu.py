"""GPU path against the UNMODIFIED reference planner compiled into oracle/_ref/libplanner_ref.so (see test_planner_ref.py):
with PC_ARITH_PCL_FLOAT the library's radiusSearch / checkSafeTrajectory values are bit-identical with the reference's, and
the reference's RRT* loops driven by the GPU grow bit-identical trees."""
import os
import subprocess

import numpy as np
import pytest

import oracle
from pointcloudtraj_b200 import PC_ARITH_PCL_FLOAT, PC_QUERY_SORTED, PcRadiusParams, PointCloudIndex, synth
from rrt_common import GOAL, PRM, START
from test_planner_ref import build_ref_check, parse_phases, two_cloud_scenario

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not oracle.have_planner_reference(), reason="needs the upstream pointcloudTraj planner compiled into oracle/_ref (make -C oracle REF=<pointcloudTraj checkout>)")]


def test_rrt_loops_driven_by_the_gpu_match_the_compiled_reference(tmp_path):
    tmp = str(tmp_path)
    exe = build_ref_check(tmp)
    p = subprocess.run([exe, two_cloud_scenario(tmp), "gpu"], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, (p.stdout, p.stderr)
    ph = parse_phases(p.stdout)
    assert len(ph) == 7 and all(v["identical"] == "1" for v in ph.values())


@pytest.mark.parametrize("prm,start", [(PRM, START), ((0.5, 0.0, 5.0, 12.0), (1.0, -2.0, 1.5))])
def test_radius_batch_pcl_float_is_bit_identical_with_compiled_radius_search(prm, start):
    pts, half = synth.forest_cloud(200_000, seed=6, variant="J", return_half=True)
    q = synth.rrt_queries(150_000, half, seed=3)
    pr = oracle.PlannerReference(*prm)
    pr.set_input(pts)
    pr.reset()
    pr.set_pt(start, GOAL, (-half, half, -half, half, 0.0, 4.0), prm[3], 100, 0.3, 0.1)
    ref = pr.radius_batch(q.astype(np.float64))
    with PointCloudIndex(max_points=len(pts)) as ix:
        ix.build(pts)
        ix.set_radius_arith(PC_ARITH_PCL_FLOAT)
        P = PcRadiusParams.make(prm[1], prm[2], prm[3], start)
        for flags in (0, PC_QUERY_SORTED):
            r = ix.radius(q, P, flags=flags)
            assert (r == ref.astype(np.float32)).all()
        # the planner's own call pattern: one double-precision point per call (tiny mapped-memory path)
        r1 = ix.radius(q[:300], P)
        assert (r1 == ref[:300].astype(np.float32)).all()


@pytest.mark.parametrize("horizon,n_traj,sample_range", [(2.0, 300, 1e6), (20.0, 80, 1e6), (20.0, 80, 6.0)])
def test_clearance_batch_vs_compiled_check_safe_trajectory(horizon, n_traj, sample_range):
    """pc_clearance_batch (PC_ARITH_PCL_FLOAT) vs the compiled checkSafeTrajectory + getPosFromBezier + checkTrajPtCol, on
    every trajectory and with NO tolerance: same verdict, same first colliding sample, same number of samples, and the same
    minimum radius (derived from the squared distances the reference's own cloud queries returned)."""
    pts, half = synth.forest_cloud(150_000, seed=6, variant="J", return_half=True)
    tr = synth.bezier_trajectories(n_traj, half * 0.9, seed=3)
    first, order, T, off, coef = tr["traj_first_seg"], tr["seg_order"], tr["seg_T"], tr["seg_coef_off"], tr["coef"]
    rng = np.random.default_rng(5)
    t_now = np.where(rng.uniform(size=n_traj) < 0.5, 0.0, rng.uniform(0, 4.0, n_traj))
    start = (0.0, 0.0, 2.0)
    pr = oracle.PlannerReference(PRM[0], PRM[1], PRM[2], sample_range)
    pr.set_input(pts)
    pr.reset()
    pr.set_pt(start, GOAL, (-half, half, -half, half, 0.0, 4.0), sample_range, 100, 0.3, 0.1)
    with PointCloudIndex(max_points=len(pts)) as ix:
        ix.build(pts)
        ix.set_radius_arith(PC_ARITH_PCL_FLOAT)
        P = PcRadiusParams.make(PRM[1], PRM[2], sample_range, start)
        fh, mr, ns = ix.clearance(first, order, T, off, coef, P, t_now=t_now, dt=0.02, horizon=horizon)
    n_hit = n_early = 0
    for t in range(n_traj):
        segs = list(range(first[t], first[t + 1]))
        ld = 3 * (int(order[segs].max()) + 1)
        mat = np.zeros((len(segs), ld))
        for r_, s in enumerate(segs):
            cc = coef[off[s]:off[s + 1]]
            mat[r_, : len(cc)] = cc
        hit, rpts, n = pr.check_safe_trajectory(order[segs], T[segs], mat, t_now[t], horizon)
        if hit:
            assert fh[t] == n - 1                       # the reference returns at its first colliding sample
            n_hit += 1
            continue
        assert fh[t] == -1 and ns[t] == n
        if n == 0:
            assert np.isinf(mr[t])
            continue
        # min over the samples of min(sqrt(d2) - search_margin, max_radius) in the reference's float32 arithmetic
        # (corridor_finder.cpp:131-132); samples that took an early-out contribute max_radius - search_margin (:115-120)
        rad = PRM[2]
        if pr.last_searched > 0:
            rad = min(float(np.sqrt(pr.last_min_d2)) - PRM[1], PRM[2])
        if pr.last_searched < n:
            rad = min(rad, PRM[2] - PRM[1])
            n_early += 1
        assert mr[t] == np.float32(rad)
    assert n_hit > 3 and n_hit < n_traj
    if sample_range < 100:
        assert n_early > 0
