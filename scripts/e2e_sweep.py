#!/usr/bin/env python
"""Sweep the PC_HOST pipeline chunk size on the bench workload (GPU box): end-to-end queries/s from pinned host memory."""
import ctypes as C
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from pointcloudtraj_b200 import PcRadiusParams, PointCloudIndex, synth  # noqa: E402

M = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
pts, half = synth.forest_cloud(1_000_000, seed=1, variant="J", return_half=True)
q = torch.from_numpy(synth.rrt_queries(M, half, seed=1000)).pin_memory()
r = torch.empty(M, dtype=torch.float32).pin_memory()
qp, rp = q.numpy(), r.numpy()
P = PcRadiusParams.make(0.25, 1.5, 30.0, (0.0, 0.0, 2.0))
print(f"# e2e pc_radius_batch PC_HOST, {M} queries, pinned buffers")
ref = None
for chunk in (1 << 19, 1 << 20, 1 << 21, 3 << 20, 1 << 22):
    os.environ["PC_HOST_CHUNK_QUERIES"] = str(chunk)
    ix = PointCloudIndex(max_points=len(pts))
    ix.build(pts)
    L = ix._L
    for _ in range(2):
        L.pc_radius_batch(ix._h, C.c_void_p(qp.ctypes.data), M, 3, 0, 0, C.byref(P), C.c_void_p(rp.ctypes.data), None)
    t0 = time.perf_counter()
    n = 6
    for _ in range(n):
        rc = L.pc_radius_batch(ix._h, C.c_void_p(qp.ctypes.data), M, 3, 0, 0, C.byref(P), C.c_void_p(rp.ctypes.data), None)
        assert rc == 0
    dt = (time.perf_counter() - t0) / n
    if ref is None:
        ref = rp.copy()
    print(f"chunk {chunk:9d}: {dt * 1e3:7.3f} ms/step  {M / dt / 1e9:6.3f} Gq/s  same={bool((rp == ref).all())}", flush=True)
    ix.close()
