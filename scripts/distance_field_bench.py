#!/usr/bin/env python
"""pc_distance_field against the composition it replaces, on the same handle, alternated call by call.

    python scripts/distance_field_bench.py [--points 1000000,5000000] [--max-ranges -1,2.0,0.5] [--reps 7] [--host-reps 3]
                                           [--out FILE]

Maps: synth.forest_cloud(n, variant="J") for every --points value.  Lattices at 0.1 m voxels centred on the map's centre:
200 x 200 x 60, 256 x 256 x 64 and 512 x 512 x 64.  For every (map, lattice, max_range; -1 = unbounded) it times, with CUDA
events on the handle's stream (torch's), the median of --reps calls after one warm-up call of each, the two alternating:
  field        pc_distance_field, PC_DEVICE: one kernel, no input array;
  composition  what a caller does today: the voxel centres made on the device with torch (the contract's fp64 expression,
               one elementwise kernel per operation, so nothing is fused, then rounded to float32), pc_knn_batch(k = 1,
               max_range) on them (pc_nearest_batch when unbounded), and the distance pass -- the winning point gathered, its
               fp64 d2 recomputed and its square root rounded to float32 (the float32 d2 that pc_knn_batch returns would not
               give the field's value bit for bit);
  knn only     the pc_knn_batch / pc_nearest_batch call of the composition alone, on the centres made beforehand: a lower
               bound of the composition's cost.
The outputs of the field and of the composition are compared bit for bit in the same run (an assertion).  A last column times
the PC_HOST call end to end (numpy outputs in pageable memory, host clock, median of --host-reps).  The card's name, power
limit and max SM clock are printed first.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LATTICES = [(200, 200, 60), (256, 256, 64), (512, 512, 64)]
VOXEL = 0.1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", default="1000000,5000000")
    ap.add_argument("--max-ranges", default="-1,2.0,0.5")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("distance_field_bench.py needs a CUDA device")
    import ctypes as C
    from pointcloudtraj_b200 import PcLattice, PointCloudIndex, synth
    from pointcloudtraj_b200 import _lib as L

    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    emit(f"# GPU: {smi[0] if smi else torch.cuda.get_device_name(0)} (name, power limit, max SM clock)")
    emit(f"# voxel {VOXEL} m, lattices centred on the map's centre; device ms per call: median [min, max] of {a.reps}, the field "
         "and the composition alternated; host ms: PC_HOST end to end")
    dev = torch.device("cuda:0")
    vp = lambda t: C.c_void_p(t.data_ptr())
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def time_once(fn):
        ev[0].record()
        fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1])

    def stat(ts):
        return f"{np.median(ts):8.3f} [{min(ts):.3f}, {max(ts):.3f}]"

    for n_points in [int(x) for x in a.points.split(",")]:
        pts, half = synth.forest_cloud(n_points, seed=3, variant="J", return_half=True)
        ix = PointCloudIndex(max_points=len(pts), device=0, stream=torch.cuda.current_stream().cuda_stream)
        ix.build(pts)
        lib = ix._L
        cloud = torch.from_numpy(pts).to(dev).double()
        fin = pts[np.isfinite(pts).all(1)]
        mid = 0.5 * (fin.min(0).astype(np.float64) + fin.max(0).astype(np.float64))
        emit(f"## map: forest J, {len(pts)} points, box {np.round(fin.min(0), 2).tolist()} .. {np.round(fin.max(0), 2).tolist()}")
        for dims in LATTICES:
            nx, ny, nz = dims
            n = nx * ny * nz
            origin = tuple(float(mid[a_] - 0.5 * dims[a_] * VOXEL) for a_ in range(3))
            lat = PcLattice.make(origin, VOXEL, dims)
            f_dist = torch.empty(n, dtype=torch.float32, device=dev)
            f_idx = torch.empty(n, dtype=torch.int32, device=dev)
            k_idx = torch.empty(n, dtype=torch.int32, device=dev)
            k_d2 = torch.empty(n, dtype=torch.float32, device=dev)
            state = {}

            def make_centres():
                ax = [(torch.arange(dims[a_], dtype=torch.float64, device=dev) + 0.5) * VOXEL + origin[a_] for a_ in range(3)]
                ax = [x.float() for x in ax]
                zz, yy, xx = torch.meshgrid(ax[2], ax[1], ax[0], indexing="ij")
                state["c"] = torch.stack([xx.reshape(-1), yy.reshape(-1), zz.reshape(-1)], 1).contiguous()

            def knn(r):
                c = state["c"]
                if r < 0:
                    rc = lib.pc_nearest_batch(ix._h, vp(c), n, 3, L.PC_DEVICE, 0, vp(k_idx), vp(k_d2))
                else:
                    rc = lib.pc_knn_batch(ix._h, vp(c), n, 3, L.PC_DEVICE, 0, 1, r, vp(k_idx), vp(k_d2))
                assert rc == L.PC_OK, lib.pc_last_error(ix._h)

            def dist_pass():
                c = state["c"].double()
                p = cloud[k_idx.clamp(min=0).long()]
                e = p - c
                d2 = (e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2]
                state["d"] = torch.where(k_idx >= 0, d2.sqrt().float(), torch.full_like(k_d2, float("inf")))

            def composition(r):
                make_centres()
                knn(r)
                dist_pass()

            def fieldcall(r):
                assert lib.pc_distance_field(ix._h, C.byref(lat), r, L.PC_DEVICE, vp(f_dist), vp(f_idx)) == L.PC_OK, \
                    lib.pc_last_error(ix._h)

            for r in [float(x) for x in a.max_ranges.split(",")]:
                fieldcall(r)
                composition(r)
                torch.cuda.synchronize()
                assert torch.equal(f_idx, k_idx), f"{dims} r={r}: indices differ from the composition"
                assert torch.equal(f_dist.view(torch.int32), state["d"].view(torch.int32)), f"{dims} r={r}: distances differ"
                tf, tc, tk = [], [], []
                for _ in range(a.reps):
                    tf.append(time_once(lambda: fieldcall(r)))
                    tc.append(time_once(lambda: composition(r)))
                    tk.append(time_once(lambda: knn(r)))
                torch.cuda.synchronize()
                assert torch.equal(f_idx, k_idx) and torch.equal(f_dist.view(torch.int32), state["d"].view(torch.int32))
                hits = float((f_idx >= 0).float().mean())
                th = []
                for _ in range(a.host_reps):
                    t0 = time.perf_counter()
                    hd, hi = ix.distance_field(origin, VOXEL, dims, None if r < 0 else r)
                    th.append((time.perf_counter() - t0) * 1e3)
                assert (hi.ravel() == f_idx.cpu().numpy()).all() and (hd.ravel().view(np.uint32) == f_dist.cpu().numpy().view(np.uint32)).all()
                emit(f"{len(pts):8d} pts {nx}x{ny}x{nz} ({n / 1e6:5.2f} M voxels) max_range={'inf' if r < 0 else r:<4} "
                     f"field {stat(tf)}  composition {stat(tc)}  knn only {stat(tk)}  speed-up {np.median(tc) / np.median(tf):5.2f}x "
                     f"(vs knn only {np.median(tk) / np.median(tf):5.2f}x)  PC_HOST {np.median(th):8.2f} ms  "
                     f"with a point {100 * hits:5.1f} %  bit-identical")
            del state
        ix.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
