#!/usr/bin/env python
"""Latency of small radius batches on the 1M-point map for the kernel / ordering choices."""
import ctypes as C, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from pointcloudtraj_b200 import PcRadiusParams, PointCloudIndex, synth, _lib
dev = torch.device("cuda", 0)
torch.cuda.set_stream(torch.cuda.Stream(device=dev))
stream = torch.cuda.current_stream().cuda_stream
pts, half = synth.forest_cloud(1_000_000, seed=1, variant="J", return_half=True)
t_pts = torch.from_numpy(pts).to(dev)
P = PcRadiusParams.make(0.25, 1.5, 30.0, (0.0, 0.0, 2.0))
print(f"{'m':>8s} {'flags':>9s} {'G':>3s} {'ms':>8s}")
for m in (1000, 4000, 8000, 16000, 32000, 50000, 100000, 200000):
    q = torch.from_numpy(synth.rrt_queries(m, half, seed=5)).to(dev)
    out = torch.empty(m, dtype=torch.float32, device=dev)
    # unsorted = a group of G lanes per query (pc_query_coop_kernel); sorted = ordered 32-query warp packets
    for flags, fname in ((2, "unsorted"), (4, "sorted")):
        for group in ((32, 16, 8) if flags == 2 else (0,)):
            os.environ["PC_QUERY_KERNEL"] = "3"
            os.environ["PC_COOP_MAX_BATCH"] = str(1 << 30)
            os.environ["PC_COOP_GROUP"] = str(group)
            ix = PointCloudIndex(max_points=len(pts), stream=stream)
            ix.build(t_pts)
            L = ix._L
            ts = []
            for _ in range(12):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                L.pc_radius_batch(ix._h, C.c_void_p(q.data_ptr()), m, 3, 1, flags, C.byref(P), C.c_void_p(out.data_ptr()), None)
                e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
            print(f"{m:8d} {fname:>9s} {group:3d} {np.median(ts[3:]):8.4f}", flush=True)
            ix.close()
