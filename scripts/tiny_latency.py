#!/usr/bin/env python
"""Latency of small blocking PC_HOST radius calls (run on the GPU box): the mapped-memory path with one warp per query (default) and
staged copies (PC_TINY_BATCH_QUERIES=0).  m = 1 is what the unmodified planner loop issues once per RRT* iteration.

    python scripts/tiny_latency.py > gpurun_out/tiny_latency.txt
"""
import ctypes as C
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from pointcloudtraj_b200 import _lib, synth
    from pointcloudtraj_b200._lib import PcRadiusParams
    L = _lib.load()
    pts, half = synth.forest_cloud(200_000, seed=6, variant="J", return_half=True)
    q = synth.rrt_queries(8192, half, seed=5)
    P = PcRadiusParams.make(0.25, 1.5, 30.0, (0.0, 0.0, 2.0))
    out = np.empty(len(q), np.float32)
    print("# blocking pc_radius_batch(PC_HOST, m) on a 200k-point map, microseconds per call (median of 5 x 400 calls, ctypes included)")
    print(f"{'m':>6s} {'warp/query':>11s} {'staged':>9s}")
    handles = {}
    names = ("warp/query", "staged")
    for name, env in zip(names, ({}, {"PC_TINY_BATCH_QUERIES": "0"})):
        os.environ.pop("PC_TINY_BATCH_QUERIES", None)
        os.environ.update(env)
        h = C.c_void_p()
        assert L.pc_index_create(C.byref(h), 0, len(pts), None) == 0
        assert L.pc_index_build(h, pts.ctypes.data_as(C.c_void_p), len(pts), 3, 0) == 0
        handles[name] = h
    for m in (1, 8, 64, 512, 4096, 8192):
        row = []
        for name in names:
            h = handles[name]
            qp, op = q.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)
            meds = []
            for rep in range(6):
                t0 = time.perf_counter()
                for _ in range(400):
                    rc = L.pc_radius_batch(h, qp, m, 3, 0, 2, C.byref(P), op, None)      # PC_HOST, PC_QUERY_UNSORTED
                meds.append((time.perf_counter() - t0) / 400 * 1e6)
                assert rc == 0
            row.append(float(np.median(meds[1:])))
        print(f"{m:6d} {row[0]:11.1f} {row[1]:9.1f}", flush=True)
    for h in handles.values():
        L.pc_index_destroy(h)


if __name__ == "__main__":
    main()
