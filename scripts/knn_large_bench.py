#!/usr/bin/env python
"""pc_knn_large_batch sweep: device-resident batches timed with CUDA events (median of repeated calls after warm-up).

    python scripts/knn_large_bench.py [--ks 33,64,128,256,512,1024] [--bound 1.0] [--order-sizes ...] [--out FILE]

Workloads:
  C1     synth.forest_cloud(200_000, variant="J"), 100 k rrt_queries
  C2     the bench map (synth.forest_cloud(1_000_000, variant="J")) at 100 k and 1 M rrt_queries
For every k and bound (unbounded, --bound m) it times the forced paths (PC_QUERY_UNSORTED: one warp per query in batch
order; PC_QUERY_SORTED: ordering pass, then the same kernel in curve order) and PC_QUERY_AUTO.  Reference lines:
pc_knn_batch at k = 32 on the same batch; for bounded runs pc_range_sorted_batch(r, max_nn = k), which gives the same rows in
CSR form (its offsets-only sizing call included, as range_sorted() makes it); scipy's cKDTree.query(k, workers=-1) on the host
for a sub-sample.  A second section times SORTED against UNSORTED on the bench map from 1 k to 1 M queries (the crossover of
PC_QUERY_AUTO).  Each line: median ms per call, [min, max] over the timed calls, queries/s of the median.  The card's name,
power limit and max SM clock are printed first.
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
    ap.add_argument("--ks", default="33,64,128,256,512,1024")
    ap.add_argument("--bound", type=float, default=1.0)
    ap.add_argument("--order-sizes", default="1000,8000,32000,100000,300000,1000000")
    ap.add_argument("--order-ks", default="33,64,256,1024")
    ap.add_argument("--scipy-queries", type=int, default=20_000)
    ap.add_argument("--skip-sweep", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("knn_large_bench.py needs a CUDA device")
    from pointcloudtraj_b200 import PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED, PointCloudIndex, synth

    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    emit(f"# GPU: {smi[0] if smi else torch.cuda.get_device_name(0)} (name, power limit, max SM clock)")
    ks = [int(s) for s in a.ks.split(",")]
    st = torch.cuda.current_stream()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, m):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        reps = int(min(15, max(5, 4e6 // max(m, 1))))
        ts = []
        for _ in range(reps):
            ev0.record(st)
            fn()
            ev1.record(st)
            ev1.synchronize()
            ts.append(ev0.elapsed_time(ev1))
        ts = np.array(ts)
        return float(np.median(ts)), float(ts.min()), float(ts.max())

    def fmt(name, m, t):
        med, lo, hi = t
        return f"{name:44s} m={m:>8d}  {med:9.4f} ms  [{lo:.4f}, {hi:.4f}]  {m / (med * 1e-3):.3e} q/s"

    def rname(r):
        return f"r={r}" if r is not None else "unbounded"

    names = {PC_QUERY_UNSORTED: "UNSORTED", PC_QUERY_SORTED: "SORTED", PC_QUERY_AUTO: "AUTO"}
    clouds = {}

    def cloud(n):
        if n not in clouds:
            pts, half = synth.forest_cloud(n, variant="J", return_half=True)
            clouds[n] = pts, half
        return clouds[n]

    def index_of(pts):
        ix = PointCloudIndex(max_points=len(pts), device=0, stream=st.cuda_stream)
        ix.build(pts)
        ix.sync()
        return ix

    if not a.skip_sweep:
        for name, n, m in (("C1", 200_000, 100_000), ("C2", 1_000_000, 100_000), ("C2", 1_000_000, 1_000_000)):
            pts, half = cloud(n)
            q = synth.rrt_queries(m, half, seed=1)
            qd = torch.from_numpy(q).cuda()
            ix = index_of(pts)
            emit(f"## {name}: forest_cloud({n}, variant='J'), half = {half:.2f} m; {m} rrt_queries(seed=1)")
            for r in (None, a.bound):
                emit(fmt(f"knn k=32 {rname(r)} AUTO (pc_knn_batch)", m, timed(lambda: ix.knn(qd, 32, r), m)))
                for k in ks:
                    for fl in (PC_QUERY_UNSORTED, PC_QUERY_SORTED, PC_QUERY_AUTO):
                        emit(fmt(f"knn_large k={k} {rname(r)} {names[fl]}", m, timed(lambda: ix.knn_large(qd, k, r, fl), m)))
                    if r is not None:
                        emit(fmt(f"range_sorted max_nn={k} {rname(r)}", m, timed(lambda: ix.range_sorted(qd, r, max_nn=k), m)))
            ix.close()
            del qd
            torch.cuda.empty_cache()
            # context: scipy's cKDTree on the host CPU, a sub-sample
            try:
                from scipy.spatial import cKDTree
                sub = q[: a.scipy_queries].astype(np.float64)
                tree = cKDTree(pts.astype(np.float64))
                for r in (None, a.bound):
                    for k in (ks[0], ks[-1]):
                        t0 = time.perf_counter()
                        tree.query(sub, k=k, workers=-1, distance_upper_bound=np.inf if r is None else r)
                        dt = time.perf_counter() - t0
                        emit(f"cKDTree k={k} {rname(r)} (host, {os.cpu_count()} logical CPUs, workers=-1) m={len(sub)}  {dt * 1e3:9.2f} ms  {len(sub) / dt:.3e} q/s")
            except ImportError:
                emit("# scipy not available")

    # the ordering crossover on the bench map
    pts, half = cloud(1_000_000)
    sizes = [int(s) for s in a.order_sizes.split(",")]
    qall = torch.from_numpy(synth.rrt_queries(max(sizes), half, seed=1)).cuda()
    ix = index_of(pts)
    emit("## ordering crossover on C2: UNSORTED ms / SORTED ms / AUTO ms (faster forced path)")
    for r in (None, a.bound):
        for k in [int(s) for s in a.order_ks.split(",")]:
            for m in sizes:
                qd = qall[:m].contiguous()
                t = {fl: timed(lambda: ix.knn_large(qd, k, r, fl), m)[0] for fl in (PC_QUERY_UNSORTED, PC_QUERY_SORTED, PC_QUERY_AUTO)}
                fast = "SORTED" if t[PC_QUERY_SORTED] < t[PC_QUERY_UNSORTED] else "UNSORTED"
                emit(f"k={k:<5d} {rname(r):9s} m={m:>8d}  {t[PC_QUERY_UNSORTED]:9.4f} {t[PC_QUERY_SORTED]:9.4f} {t[PC_QUERY_AUTO]:9.4f}  faster={fast}")
    ix.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
