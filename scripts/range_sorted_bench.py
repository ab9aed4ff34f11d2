#!/usr/bin/env python
"""pc_range_sorted_batch on the range workloads of scripts/range_ab.py: device buffers, CUDA events, median and spread.

    python scripts/range_sorted_bench.py [--reps 15] [--out profiles/r5_range_sorted.txt]

Workloads (seeded): C1 = 200 k-point forest J (seed 6), 100 k rrt_queries (seed 7), r = 1 m; and 50 k rrt_queries (seed 2) on
the 1 M-point map (forest J, seed 1), r = 1 m.  For max_nn in {0, 16, 64, 256} the sorted call is timed alternately with
pc_range_batch on the same inputs (one call of each per round), and pc_knn_batch(k = max_nn, r) next to it for max_nn <= 32.
Every call includes its one host synchronisation (the read-back of the total).  A torch.profiler pass over the C1 max_nn = 0
call lists the kernel times.  Host CPU context: scipy cKDTree.query(k = max_nn, distance_upper_bound = r, workers = -1) for
the capped cases, query_ball_point + an fp64 sort by (d2, index) on the host for max_nn = 0.  The card's name, power limit
and max SM clock are printed first.
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MAX_NN = (0, 16, 64, 256)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("range_sorted_bench.py needs a CUDA device")
    from pointcloudtraj_b200 import _lib, synth
    from pointcloudtraj_b200 import PointCloudIndex
    lib = _lib.load()
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    emit(f"# GPU: {smi[0] if smi else torch.cuda.get_device_name(0)} (name, power limit, max SM clock)")
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream()
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def once(fn):
        ev0.record(st)
        fn()
        ev1.record(st)
        ev1.synchronize()
        return ev0.elapsed_time(ev1)

    def stats(ts):
        ts = np.array(ts)
        return f"{np.median(ts):8.3f} ms [{ts.min():.3f}, {ts.max():.3f}]"

    for name, n_pts, pseed, n_q, qseed in (("C1", 200_000, 6, 100_000, 7), ("1M map", 1_000_000, 1, 50_000, 2)):
        pts, half = synth.forest_cloud(n_pts, seed=pseed, variant="J", return_half=True)
        q = synth.rrt_queries(n_q, half, seed=qseed)
        r = 1.0
        emit(f"## {name}: forest_cloud({n_pts}, seed={pseed}, variant='J'), rrt_queries({n_q}, seed={qseed}), r = {r} m, "
             f"{a.reps} alternated rounds, median [min, max]")
        ix = PointCloudIndex(max_points=n_pts, device=0, stream=st.cuda_stream)
        ix.build(pts)
        ix.sync()
        h, m = ix._h, n_q
        tq = torch.from_numpy(q).to(dev)
        tr = torch.full((1,), r, dtype=torch.float64, device=dev)
        off = torch.empty(m + 1, dtype=torch.int64, device=dev)
        assert lib.pc_range_batch(h, vp(tq), m, 3, 1, vp(tr), 1, vp(off), None, 0) == 0
        total = int(off[-1].item())
        lst = torch.empty(total, dtype=torch.int32, device=dev)
        sidx = torch.empty(total, dtype=torch.int32, device=dev)
        sd2 = torch.empty(total, dtype=torch.float32, device=dev)
        soff = torch.empty(m + 1, dtype=torch.int64, device=dev)
        sizes = np.diff(off.cpu().numpy())
        emit(f"hits {total} ({total / m:.1f} per query), lists > 512: {(sizes > 512).sum()}, longest {sizes.max()}")
        rng_call = lambda: lib.pc_range_batch(h, vp(tq), m, 3, 1, vp(tr), 1, vp(off), vp(lst), total)
        for max_nn in MAX_NN:
            srt_call = lambda: lib.pc_range_sorted_batch(h, vp(tq), m, 3, 1, vp(tr), 1, max_nn, vp(soff), vp(sidx), vp(sd2), total)
            calls = [("pc_range_batch", rng_call), (f"pc_range_sorted_batch max_nn={max_nn}", srt_call)]
            if 0 < max_nn <= 32:
                kidx = torch.empty(m * max_nn, dtype=torch.int32, device=dev)
                kd2 = torch.empty(m * max_nn, dtype=torch.float32, device=dev)
                calls.append((f"pc_knn_batch k={max_nn} r={r}", lambda: lib.pc_knn_batch(h, vp(tq), m, 3, 1, 0, max_nn, r, vp(kidx), vp(kd2))))
            for _, fn in calls:            # warm-up
                for _ in range(2):
                    assert fn() == 0
            torch.cuda.synchronize()
            ts = {c[0]: [] for c in calls}
            for _ in range(a.reps):
                for cname, fn in calls:
                    ts[cname].append(once(fn))
            for cname, _ in calls:
                emit(f"{cname:40s} {stats(ts[cname])}")
            if max_nn == 0:
                assert (soff == off).all().item(), "offsets differ from pc_range_batch"
        if name == "C1":
            # where the time of the max_nn = 0 call goes, per kernel (a separate, profiled run)
            from torch.profiler import ProfilerActivity, profile
            call = lambda: lib.pc_range_sorted_batch(h, vp(tq), m, 3, 1, vp(tr), 1, 0, vp(soff), vp(sidx), vp(sd2), total)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    call()
                torch.cuda.synchronize()
            emit("### kernels of pc_range_sorted_batch max_nn=0 (torch.profiler, 5 calls, per-call mean)")
            for e in sorted(prof.key_averages(), key=lambda e: -e.device_time_total):
                if e.device_time_total > 0:
                    emit(f"  {e.key[:70]:70s} {e.device_time_total / 5 / 1e3:8.3f} ms  x{e.count // 5}")
        ix.close()
        # host CPU context
        try:
            from scipy.spatial import cKDTree
        except ImportError:
            emit("scipy not available")
            continue
        tree = cKDTree(pts.astype(np.float64))
        for max_nn in MAX_NN:
            t0 = time.perf_counter()
            if max_nn == 0:
                lists = tree.query_ball_point(q.astype(np.float64), r, workers=-1)
                cnt = np.array([len(x) for x in lists])
                ids = np.concatenate([np.asarray(x, np.int64) for x in lists])
                row = np.repeat(np.arange(m), cnt)
                d = pts[ids].astype(np.float64) - q[row].astype(np.float64)
                s = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
                np.lexsort((ids, s, row))
            else:
                tree.query(q.astype(np.float64), k=max_nn, distance_upper_bound=r, workers=-1)
            dt = time.perf_counter() - t0
            what = "query_ball_point + host fp64 sort" if max_nn == 0 else f"query k={max_nn} distance_upper_bound={r}"
            emit(f"scipy cKDTree {what:40s} {dt * 1e3:9.1f} ms  ({os.cpu_count()} logical CPUs, workers=-1)")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
