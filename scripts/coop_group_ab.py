#!/usr/bin/env python
"""Mid-size unordered batches (C2's own 50 k RRT* samples and around): one thread per query against a group of 8 lanes per
query (pc_query_coop_kernel).  Device buffers, CUDA events around the call, median of 8; results compared."""
import ctypes as C, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from pointcloudtraj_b200 import PcRadiusParams, PointCloudIndex, synth
dev = torch.device("cuda", 0)
torch.cuda.set_stream(torch.cuda.Stream(device=dev))
stream = torch.cuda.current_stream().cuda_stream
pts, half = synth.forest_cloud(1_000_000, seed=1, variant="J", return_half=True)
t_pts = torch.from_numpy(pts).to(dev)
P = PcRadiusParams.make(0.25, 1.5, 30.0, (0.0, 0.0, 2.0))
handles = {}
for name, env in (("thread", {"PC_COOP_MAX_BATCH": "0"}), ("g8", {"PC_COOP_MAX_BATCH": "100000000", "PC_COOP_GROUP": "8"}),
                  ("auto", {})):
    for k in ("PC_COOP_MAX_BATCH", "PC_COOP_GROUP"):
        os.environ.pop(k, None)
    os.environ.update(env)
    handles[name] = PointCloudIndex(max_points=len(pts), stream=stream)
    handles[name].build(t_pts)
print(f"{'m':>8s} {'kind':>8s} " + " ".join(f"{n:>9s}" for n in handles) + "   ms (PC_QUERY_UNSORTED; auto = the library's own choice)")
for m in (8_000, 16_000, 24_000, 32_000, 50_000, 100_000, 200_000, 400_000, 800_000):
    q = torch.from_numpy(synth.rrt_queries(m, half, seed=5)).to(dev)
    for kind in ("radius", "nearest"):
        row, ref = [], None
        for name, ix in handles.items():
            out = torch.empty(m, dtype=torch.float32, device=dev)
            oi = torch.empty(m, dtype=torch.int32, device=dev)
            flags = 0 if name == "auto" else 2
            ts = []
            for _ in range(11):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                if kind == "radius":
                    rc = ix._L.pc_radius_batch(ix._h, C.c_void_p(q.data_ptr()), m, 3, 1, flags, C.byref(P), C.c_void_p(out.data_ptr()), None)
                else:
                    rc = ix._L.pc_nearest_batch(ix._h, C.c_void_p(q.data_ptr()), m, 3, 1, flags, C.c_void_p(oi.data_ptr()), C.c_void_p(out.data_ptr()))
                assert rc == 0
                e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
            row.append(float(np.median(ts[3:])))
            if ref is None:
                ref = (out.clone(), oi.clone())
            else:
                assert bool((out == ref[0]).all()) and (kind == "radius" or bool((oi == ref[1]).all())), name
        print(f"{m:8d} {kind:>8s} " + " ".join(f"{v:9.4f}" for v in row), flush=True)
