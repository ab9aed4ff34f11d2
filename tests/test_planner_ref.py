"""Parity of the planner-side restatements against the UNMODIFIED reference planner sources, compiled by oracle/Makefile
into oracle/_ref/libplanner_ref.so (Planner/src/corridor_finder.cpp as a whole; Planner/src/sim_planning_demo.cpp:715-781
cut out at build time) on stand-in Eigen / pcl / ros headers (oracle/shim).  CPU only.

* include/pc_rrt.hpp (reference-quirks mode) reproduces SafeRegionExpansion / SafeRegionRefine / SafeRegionEvaluate /
  treeRepair bit for bit: corridor, radii and the whole node list after every phase.
* oracle/planner_oracle.c (the restatement the GPU tests use at scale) agrees with the compiled getPosFromBezier /
  checkSafeTrajectory / radiusSearch.
"""
import os
import subprocess

import numpy as np
import pytest

import oracle
from pointcloudtraj_b200 import synth
from rrt_common import GOAL, PRM, START, blocked_cloud, write_input

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.skipif(not oracle.have_planner_reference(), reason="needs the upstream pointcloudTraj planner compiled into oracle/_ref (make -C oracle REF=<pointcloudTraj checkout>)")


def build_ref_check(tmp):
    exe = os.path.join(tmp, "rrt_ref_check")
    rdir, pdir = os.path.join(ROOT, "oracle", "_ref"), os.path.join(ROOT, "pointcloudtraj_b200")
    subprocess.run(["g++", "-std=c++14", "-O2", "-ffp-contract=off", "-o", exe, os.path.join(ROOT, "tests", "c", "rrt_ref_check.cpp"),
                    "-I", os.path.join(ROOT, "include"), "-L", rdir, "-lplanner_ref", "-L", pdir, "-lpcindex",
                    f"-Wl,-rpath,{rdir}", f"-Wl,-rpath,{pdir}"], check=True, capture_output=True)
    return exe


def two_cloud_scenario(tmp, n_points=60_000, max_iter=6000, refine_iter=1500):
    """Growth on a forest map, then a second cloud message that puts new obstacles on two spheres of the reference's own
    corridor (so SafeRegionEvaluate has to drop them and treeRepair runs)."""
    pts, half = synth.forest_cloud(n_points, seed=6, variant="J", return_half=True)
    half = max(half, 12.0)
    pr = oracle.PlannerReference(*PRM)
    pr.set_input(pts)
    pr.reset()
    pr.set_pt(START, GOAL, (-half, half, -half, half, 0.0, 4.0), PRM[3], max_iter, 0.3, 0.1)
    pr.expand(max_iter)
    p, r = pr.path()
    assert pr.stats()["path_exists"] and len(r) >= 5
    pts2 = blocked_cloud(pts, [p[len(p) // 2], p[len(p) // 3]])
    path = os.path.join(tmp, "in.bin")
    write_input(path, pts, half, max_iter=max_iter, K=128, pts2=pts2, refine_iter=refine_iter)
    return path


def parse_phases(stdout):
    out = {}
    for ln in stdout.splitlines():
        f = ln.split()
        out[f[0]] = dict(kv.split("=") for kv in f[1:])
    return out


def test_rrt_driver_reproduces_compiled_reference_bit_for_bit(tmp_path):
    tmp = str(tmp_path)
    exe = build_ref_check(tmp)
    p = subprocess.run([exe, two_cloud_scenario(tmp), "ref"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, (p.stdout, p.stderr)
    ph = parse_phases(p.stdout)
    assert list(ph) == ["expand", "refine1", "evaluate1", "refine2", "evaluate2", "refine3", "evaluate3"]
    assert all(v["identical"] == "1" for v in ph.values())
    assert int(ph["expand"]["nodes"].split("/")[0]) > 100 and int(ph["expand"]["path"].split("/")[0]) >= 5
    # the second cloud really exercised SafeRegionEvaluate + treeRepair: nodes were deleted, then the tree grew again
    assert int(ph["evaluate1"]["nodes"].split("/")[0]) < int(ph["refine1"]["nodes"].split("/")[0])
    assert int(ph["refine3"]["nodes"].split("/")[0]) > int(ph["evaluate1"]["nodes"].split("/")[0])


def test_oracle_radius_search_vs_compiled_reference():
    """oracle radiusSearch (fp64 epilogue on the kd-tree's fp64 d2) vs the compiled corridor_finder.cpp:113-133 (d2 through
    PCL's float32 interface): within 1e-6 relative of the obstacle distance, and bit-identical once the oracle's d2 is pushed
    through the same float32 rounding + float32 sqrt."""
    pts, half = synth.forest_cloud(50_000, seed=6, variant="J", return_half=True)
    q = synth.rrt_queries(20_000, half, seed=3)
    qd = q.astype(np.float64) + np.random.default_rng(0).uniform(-1e-9, 1e-9, q.shape)     # genuine double-precision points
    for prm, start in ((PRM, START), ((0.5, 0.0, 2.0, 5.0), (1.0, -2.0, 1.5))):
        pr = oracle.PlannerReference(*prm)
        pr.set_input(pts)
        pr.reset()
        pr.set_pt(start, GOAL, (-half, half, -half, half, 0.0, 4.0), prm[3], 100, 0.3, 0.1)
        ref = pr.radius_batch(qd)
        ko = oracle.KdOracle().build(pts)
        P = oracle.RadiusParams.make(prm[1], prm[2], prm[3], start)
        mine = np.array([ko.radius_search(P, p)[0] for p in qd[:4000]])
        assert (np.abs(mine - ref[:4000]) <= 1e-6 * (np.abs(ref[:4000]) + prm[1]) + 1e-12).all()
        # the float32 path, from the oracle's exact nearest distance
        _, d2 = ko.nearest(qd.astype(np.float32))
        rad = np.minimum(np.sqrt(d2.astype(np.float32)).astype(np.float64) - prm[1], prm[2])
        far = np.sqrt(((qd - np.array(start)) ** 2).sum(1)) > prm[3] + prm[2]
        rad[far] = prm[2] - prm[1]
        assert (~far).any() and (far.any() or prm is PRM)          # the second set has queries beyond the sensing range
        assert (rad == ref).all()


def test_oracle_bezier_and_clearance_walk_vs_compiled_reference():
    """po_bezier_pos / po_check_safe_trajectory (oracle/planner_oracle.c) vs the compiled getPosFromBezier /
    checkSafeTrajectory: positions bit-identical, the sampled points (float32) identical, same verdict and same first hit."""
    rng = np.random.default_rng(1)
    pr = oracle.PlannerReference(*PRM)
    for order in range(3, 13):
        c = rng.normal(size=3 * (order + 1)) * 5
        for u in (0.0, 1.0, 0.5, 1e-300, *rng.uniform(size=20)):
            assert (oracle.bezier_pos(c, order, u) == pr.bezier_pos(c, order, u)).all()
    pts, half = synth.forest_cloud(80_000, seed=6, variant="J", return_half=True)
    pr.set_input(pts)
    pr.reset()
    pr.set_pt(START, GOAL, (-half, half, -half, half, 0.0, 4.0), PRM[3], 100, 0.3, 0.1)
    ko = oracle.KdOracle().build(pts)
    P = oracle.RadiusParams.make(PRM[1], PRM[2], PRM[3], START)
    tr = synth.bezier_trajectories(120, half * 0.9, seed=3)
    first, order, T, off, coef = tr["traj_first_seg"], tr["seg_order"], tr["seg_T"], tr["seg_coef_off"], tr["coef"]
    t_now = np.where(rng.uniform(size=120) < 0.5, 0.0, rng.uniform(0, 4.0, 120))
    n_hit = 0
    for horizon in (2.0, 20.0):
        for t in range(len(first) - 1):
            segs = list(range(first[t], first[t + 1]))
            ld = 3 * (int(order[segs].max()) + 1)
            mat = np.zeros((len(segs), ld))
            for r_, s in enumerate(segs):
                cc = coef[off[s]:off[s + 1]]
                mat[r_, : len(cc)] = cc
            hit, rpts, n = pr.check_safe_trajectory(order[segs], T[segs], mat, t_now[t], horizon)
            mine = ko.check_safe_trajectory(P, order[segs], T[segs], mat, t_now=float(t_now[t]), stop_time=horizon, cap=8192)
            borderline = np.abs(mine["radius"]).min() < 1e-6 if len(mine["radius"]) else False
            if borderline:
                continue
            assert hit == (mine["first_hit"] >= 0)
            k = mine["first_hit"] + 1 if hit else mine["n_samples"]          # the reference stops at the first colliding sample
            assert n == k and (rpts == mine["pts"][:k]).all()
            n_hit += hit
    assert n_hit > 5


@pytest.mark.parametrize("goal,inlier", [(0.15, 0.3), (0.0, 0.5), (0.6, 0.2), (1.0, 0.0)])
def test_oracle_sample_stream_vs_compiled_reference(goal, inlier):
    """po_gen_samples (minstd_rand0 + libstdc++'s generate_canonical restated in C) against k calls of the unmodified genSample
    (corridor_finder.cpp:333-383) on the planner's own engine: bit-identical samples, and the stream continues from the
    returned engine state."""
    start, end, box = (0.0, 0.0, 2.0), (40.0, 10.0, 2.0), (-50.0, 50.0, -50.0, 50.0, 0.0, 5.0)
    ref = oracle.PlannerReference(0.6, 0.25, 1.5, 30.0)
    ref.set_pt(start, end, box, 30.0, 1000, inlier, goal)
    want = ref.gen_samples(300_000)
    s = oracle.Sampler.make(start, end, box, 30.0, 0.6, inlier, goal)
    got = oracle.gen_samples(s, 100_000)
    got2 = oracle.gen_samples(s, 200_000)
    assert (got == want[:100_000]).all() and (got2 == want[100_000:]).all()
    share = (want == np.array(end)).all(1).mean()
    assert abs(share - goal) < 0.01
