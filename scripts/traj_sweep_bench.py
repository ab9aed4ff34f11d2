#!/usr/bin/env python
"""pc_trajectory_sweep_batch timings: device-resident batches timed with CUDA events (median of repeated calls after warm-up).

    python scripts/traj_sweep_bench.py [--points 5000000] [--n-traj 10000] [--radii 0.1,0.3,0.5] [--tols 1e-2,1e-3,1e-4]
                                       [--reps 5] [--out FILE]

Workload (the C4 size): synth.forest_cloud(--points, variant="J"), --n-traj trajectories of synth.bezier_trajectories with
orders 1..12, horizon 2 s, t_now 0.  For every (r, tol) it times the sweep and, on the same trajectories, pc_clearance_batch at
dt 0.02 (search_margin r, max_radius 1.5, sample_range < 0), and reports how many trajectories have a contact.  A last line
times one blocking PC_HOST call of a single 5-segment order-5 trajectory (the planner's pattern), host clock, median of 200.
The card's name, power limit and max / current SM clock are printed first.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=5_000_000)
    ap.add_argument("--n-traj", type=int, default=10_000)
    ap.add_argument("--radii", default="0.1,0.3,0.5")
    ap.add_argument("--tols", default="1e-2,1e-3,1e-4")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("traj_sweep_bench.py needs a CUDA device")
    import ctypes as C
    from pointcloudtraj_b200 import PcRadiusParams, PointCloudIndex, synth
    from pointcloudtraj_b200 import _lib as L

    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    emit(f"# GPU: {smi[0] if smi else torch.cuda.get_device_name(0)} (name, power limit, max SM clock, current SM clock)")
    pts, half = synth.forest_cloud(a.points, seed=3, variant="J", return_half=True)
    ix = PointCloudIndex(max_points=len(pts), device=0, stream=torch.cuda.current_stream().cuda_stream)
    ix.build(pts)
    tr = synth.bezier_trajectories(a.n_traj, half * 0.9, seed=8, order_range=(1, 12))
    n = a.n_traj
    rec = np.zeros(n, dtype=np.dtype([("first_seg", "<i4"), ("num_seg", "<i4"), ("t_now", "<f8")]))
    rec["first_seg"], rec["num_seg"] = tr["traj_first_seg"][:-1], np.diff(tr["traj_first_seg"])
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    d_rec, d_order, d_T = dev(rec.view(np.uint8)), dev(tr["seg_order"].astype(np.int32)), dev(tr["seg_T"])
    d_off, d_coef = dev(tr["seg_coef_off"].astype(np.int64)), dev(tr["coef"])
    d_seg, d_s, d_idx = torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda"), \
        torch.empty(n, dtype=torch.int32, device="cuda")
    d_fh, d_mr = torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.float32, device="cuda")
    vp = lambda t: C.c_void_p(t.data_ptr())
    n_seg, n_coef = len(tr["seg_order"]), len(tr["coef"])
    lib = ix._L
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(a.reps):
            ev0.record()
            fn()
            ev1.record()
            torch.cuda.synchronize()
            ts.append(ev0.elapsed_time(ev1))
        return float(np.median(ts)), min(ts), max(ts)

    emit(f"# {len(pts)} points, {n} trajectories, {n_seg} segments (orders 1..12), horizon 2 s; ms per call: median [min, max]")
    for r in [float(x) for x in a.radii.split(",")]:
        params = PcRadiusParams.make(r, 1.5, -1.0, (0.0, 0.0, 0.0))
        clr = lambda: lib.pc_clearance_batch(ix._h, vp(d_rec), n, vp(d_order), vp(d_T), vp(d_off), n_seg, vp(d_coef), n_coef,
                                             L.PC_DEVICE, 0.02, 2.0, C.byref(params), vp(d_fh), vp(d_mr), C.c_void_p(0))
        mc, lo_c, hi_c = timed(clr)
        hits_c = int((d_fh >= 0).sum())
        for tol in [float(x) for x in a.tols.split(",")]:
            sw = lambda: lib.pc_trajectory_sweep_batch(ix._h, vp(d_rec), n, vp(d_order), vp(d_T), vp(d_off), n_seg, vp(d_coef),
                                                       n_coef, L.PC_DEVICE, 2.0, r, tol, vp(d_seg), vp(d_s), vp(d_idx))
            assert sw() == L.PC_OK
            ms, lo, hi = timed(sw)
            hits = int((d_seg >= 0).sum())
            emit(f"r={r:<4} tol={tol:<6g} sweep {ms:9.3f} ms [{lo:.3f}, {hi:.3f}] contacts {hits:6d} | "
                 f"clearance dt=0.02 {mc:8.3f} ms [{lo_c:.3f}, {hi_c:.3f}] first hits {hits_c:6d}")
    one = synth.bezier_trajectories(1, half * 0.9, seed=77, order_range=(5, 5), seg_range=(5, 5))
    args = (one["traj_first_seg"], one["seg_order"], one["seg_T"], one["seg_coef_off"], one["coef"], 0.3, 1e-3)
    for _ in range(20):
        ix.trajectory_sweep(*args)
    ts = []
    for _ in range(200):
        t0 = time.perf_counter()
        ix.trajectory_sweep(*args)
        ts.append((time.perf_counter() - t0) * 1e3)
    res = ix.trajectory_sweep(*args)
    emit(f"single trajectory (5 segments, order 5, r=0.3, tol=1e-3), blocking PC_HOST call incl. the Python wrapper: "
         f"median {np.median(ts):.3f} ms [min {min(ts):.3f}, p90 {np.percentile(ts, 90):.3f}]; contact seg {int(res[0][0])}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    ix.close()


if __name__ == "__main__":
    main()
