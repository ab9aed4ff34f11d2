#!/usr/bin/env python
"""pc_trajectory_nearest_batch timings: device-resident batches timed with CUDA events (median of repeated calls after warm-up).

    python scripts/traj_nearest_bench.py [--points 5000000] [--n-traj 10000] [--max-ranges -1,0.5,1.5] [--tols 1e-2,1e-3,1e-4]
                                         [--reps 5] [--out FILE]

Workload (the C4 size): synth.forest_cloud(--points, variant="J"), --n-traj trajectories of synth.bezier_trajectories with
orders 1..12, horizon 2 s, t_now 0.  For every (max_range, tol) it times the call and reports how many rows have a witness and
their median d.  On the same trajectories it times pc_clearance_batch at dt 0.02 (max_radius 1.5, sample_range < 0) and, per
tol, what a caller does today to get the same number from pc_trajectory_sweep_batch: bisect the radius on [0, 1.5] until the
bracket is tol wide (sweep tol = tol / 4; a contact at r moves the top to r + tol / 4, none moves the bottom to r).  One call
takes one radius for the whole batch, so a per-trajectory bisection needs at least that many calls; the bisection of the
batch's median clearance is timed call by call and summed, a lower bound of the caller's cost.  A last line times one
blocking PC_HOST call of a single 5-segment order-5 trajectory (the planner's pattern), host clock, median of 200.  The
card's name, power limit and max / current SM clock are printed first.
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
    ap.add_argument("--max-ranges", default="-1,0.5,1.5")
    ap.add_argument("--tols", default="1e-2,1e-3,1e-4")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("traj_nearest_bench.py needs a CUDA device")
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
    i32 = lambda: torch.empty(n, dtype=torch.int32, device="cuda")
    f64 = lambda: torch.empty(n, dtype=torch.float64, device="cuda")
    d_seg, d_s, d_idx, d_dist = i32(), f64(), i32(), f64()
    d_fh, d_mr = i32(), torch.empty(n, dtype=torch.float32, device="cuda")
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

    def nearest(max_range, tol):
        return lambda: lib.pc_trajectory_nearest_batch(ix._h, vp(d_rec), n, vp(d_order), vp(d_T), vp(d_off), n_seg, vp(d_coef),
                                                       n_coef, L.PC_DEVICE, 2.0, max_range, tol, vp(d_seg), vp(d_s), vp(d_idx),
                                                       vp(d_dist))

    def sweep(r, tol):
        return lambda: lib.pc_trajectory_sweep_batch(ix._h, vp(d_rec), n, vp(d_order), vp(d_T), vp(d_off), n_seg, vp(d_coef),
                                                     n_coef, L.PC_DEVICE, 2.0, r, tol, vp(d_seg), vp(d_s), vp(d_idx))

    emit(f"# {len(pts)} points, {n} trajectories, {n_seg} segments (orders 1..12), horizon 2 s; ms per call: median [min, max]")
    params = PcRadiusParams.make(0.0, 1.5, -1.0, (0.0, 0.0, 0.0))
    clr = lambda: lib.pc_clearance_batch(ix._h, vp(d_rec), n, vp(d_order), vp(d_T), vp(d_off), n_seg, vp(d_coef), n_coef,
                                         L.PC_DEVICE, 0.02, 2.0, C.byref(params), vp(d_fh), vp(d_mr), C.c_void_p(0))
    mc, lo_c, hi_c = timed(clr)
    emit(f"pc_clearance_batch dt=0.02 (max_radius 1.5) {mc:8.3f} ms [{lo_c:.3f}, {hi_c:.3f}]; "
         f"median sampled clearance {float(d_mr.median()):.4f} m")
    for tol in [float(x) for x in a.tols.split(",")]:
        med = None
        for mr in [float(x) for x in a.max_ranges.split(",")]:
            assert nearest(mr, tol)() == L.PC_OK
            ms, lo, hi = timed(nearest(mr, tol))
            dist = d_dist.cpu().numpy()
            found = np.isfinite(dist)
            if mr < 0:
                med = float(np.median(dist[found]))
            emit(f"tol={tol:<6g} max_range={mr:<4g} nearest {ms:9.3f} ms [{lo:.3f}, {hi:.3f}] witnesses {int(found.sum()):6d} "
                 f"median d {float(np.median(dist[found])) if found.any() else float('nan'):.4f} m")
        # the bisection of the median clearance on [0, 1.5] with the sweep
        blo, bhi, total, calls = 0.0, 1.5, 0.0, 0
        while bhi - blo > tol:
            r = 0.5 * (blo + bhi)
            ms, _, _ = timed(sweep(r, tol / 4))
            total += ms
            calls += 1
            if med <= r:
                bhi = min(bhi, r + tol / 4)
            else:
                blo = r
        emit(f"tol={tol:<6g} bisection over pc_trajectory_sweep_batch on [0, 1.5]: {calls} calls, {total:9.3f} ms in all "
             f"(mean call {total / calls:.3f} ms)")
    one = synth.bezier_trajectories(1, half * 0.9, seed=77, order_range=(5, 5), seg_range=(5, 5))
    args = (one["traj_first_seg"], one["seg_order"], one["seg_T"], one["seg_coef_off"], one["coef"], 1e-3)
    for _ in range(20):
        ix.trajectory_nearest(*args, max_range=1.5)
    ts = []
    for _ in range(200):
        t0 = time.perf_counter()
        ix.trajectory_nearest(*args, max_range=1.5)
        ts.append((time.perf_counter() - t0) * 1e3)
    res = ix.trajectory_nearest(*args, max_range=1.5)
    emit(f"single trajectory (5 segments, order 5, max_range=1.5, tol=1e-3), blocking PC_HOST call incl. the Python wrapper: "
         f"median {np.median(ts):.3f} ms [min {min(ts):.3f}, p90 {np.percentile(ts, 90):.3f}]; d {float(res[3][0]):.4f}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    ix.close()


if __name__ == "__main__":
    main()
