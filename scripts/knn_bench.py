#!/usr/bin/env python
"""pc_knn_batch sweep on the bench map: device-resident batches timed with CUDA events after warm-up.

    python scripts/knn_bench.py [--sizes 1000,8000,...] [--ks 1,2,4,8,16,32] [--out FILE]

Cloud and queries are bench.py's (C2 map: synth.forest_cloud(1_000_000, variant="J"), synth.rrt_queries).  For every batch
size, k and bound (unbounded, 1.75 m) it times the two forced paths (PC_QUERY_UNSORTED: one warp per query;
PC_QUERY_SORTED: ordering pass + 32-query packets) and PC_QUERY_AUTO, plus pc_nearest_batch on the same batch as the k = 1
reference line.  Each line: median ms per call, [min, max] over the timed calls, queries/s of the median.  scipy's cKDTree
(workers=-1, host CPU) on a sub-sample gives context.  The card's name, power limit and max SM clock are printed first.
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
    ap.add_argument("--sizes", default="1000,8000,64000,512000,2000000,10000000")
    ap.add_argument("--ks", default="1,2,4,8,16,32")
    ap.add_argument("--bound", type=float, default=1.75)
    ap.add_argument("--scipy-queries", type=int, default=100_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("knn_bench.py needs a CUDA device")
    from pointcloudtraj_b200 import PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED, PointCloudIndex, synth

    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    emit(f"# GPU: {smi[0] if smi else torch.cuda.get_device_name(0)} (name, power limit, max SM clock)")
    sizes = [int(s) for s in a.sizes.split(",")]
    ks = [int(s) for s in a.ks.split(",")]
    pts, half = synth.forest_cloud(1_000_000, variant="J", return_half=True)
    qall = synth.rrt_queries(max(sizes), half, seed=1)
    emit(f"# cloud: forest_cloud(1_000_000, variant='J'), half = {half:.2f} m; queries: rrt_queries(seed=1), first m of {len(qall)}")
    st = torch.cuda.current_stream()
    ix = PointCloudIndex(max_points=len(pts), device=0, stream=st.cuda_stream)
    ix.build(pts)
    ix.sync()
    qd_all = torch.from_numpy(qall).cuda()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, m):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        reps = int(min(20, max(5, 4e6 // max(m, 1))))
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
        return f"{name:34s} m={m:>9d}  {med:9.4f} ms  [{lo:.4f}, {hi:.4f}]  {m / (med * 1e-3):.3e} q/s"

    names = {PC_QUERY_UNSORTED: "UNSORTED", PC_QUERY_SORTED: "SORTED", PC_QUERY_AUTO: "AUTO"}
    summary = []
    for m in sizes:
        qd = qd_all[:m].contiguous()
        emit(f"## m = {m}")
        tn = timed(lambda: ix.nearest(qd), m)
        emit(fmt("pc_nearest_batch", m, tn))
        for r in (None, a.bound):
            for k in ks:
                res = {}
                for fl in (PC_QUERY_UNSORTED, PC_QUERY_SORTED, PC_QUERY_AUTO):
                    res[fl] = timed(lambda: ix.knn(qd, k, r, fl), m)
                    emit(fmt(f"knn k={k:<2d} {'r=' + str(r) if r is not None else 'unbounded':9s} {names[fl]}", m, res[fl]))
                fast = min((PC_QUERY_UNSORTED, PC_QUERY_SORTED), key=lambda f: res[f][0])
                summary.append((m, k, r, names[fast], res[PC_QUERY_UNSORTED][0], res[PC_QUERY_SORTED][0], res[PC_QUERY_AUTO][0]))
        del qd
        torch.cuda.empty_cache()
    emit("## faster forced path per (m, k, bound): UNSORTED ms / SORTED ms / AUTO ms")
    for m, k, r, f, u, s, au in summary:
        emit(f"m={m:>9d} k={k:<2d} {'r=' + str(r) if r is not None else 'unbounded':9s} faster={f:8s} {u:9.4f} {s:9.4f} {au:9.4f}")
    # context: scipy's cKDTree on the host CPU
    try:
        from scipy.spatial import cKDTree
        sub = qall[: a.scipy_queries]
        t0 = time.perf_counter()
        tree = cKDTree(pts.astype(np.float64))
        tb = time.perf_counter() - t0
        emit(f"## scipy cKDTree (host CPU, {os.cpu_count()} logical CPUs, workers=-1), build {tb:.3f} s, {len(sub)} queries")
        for r in (None, a.bound):
            for k in ks:
                t0 = time.perf_counter()
                tree.query(sub, k=k, workers=-1, distance_upper_bound=np.inf if r is None else r)
                dt = time.perf_counter() - t0
                emit(f"cKDTree k={k:<2d} {'r=' + str(r) if r is not None else 'unbounded':9s} m={len(sub)}  {dt * 1e3:9.2f} ms  {len(sub) / dt:.3e} q/s")
    except ImportError:
        emit("## scipy not available")
    ix.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
