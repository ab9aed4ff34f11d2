#!/usr/bin/env python
"""A/B of libpcindex variants (build/variants/lib_*.so, see scripts/variants_ab.py build) on the range workloads:
C1 (200 k points, 100 k queries, r = 1 m) and 50 k queries on the 1 M-point map; device buffers, CUDA events, median of 7.
Each workload times pc_range_batch and pc_range_sorted_batch at max_nn 0 and 64 (with d2).  `same`: offsets, indices and d2
of every call are bit-identical with those of the first library.

    python scripts/range_ab.py [--rounds N]      # N rounds, every library once per round, in turn
"""
import argparse
import ctypes as C
import glob
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=1)
    a = ap.parse_args()
    import torch
    from pointcloudtraj_b200 import _lib, synth
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(f"# GPU: {smi.splitlines()[0] if smi else torch.cuda.get_device_name(0)} (name, power limit)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_stream(torch.cuda.Stream(device=dev))
    stream = torch.cuda.current_stream().cuda_stream
    cases = []
    for n_pts, n_q, seed in ((200_000, 100_000, 6), (1_000_000, 50_000, 1)):
        pts, half = synth.forest_cloud(n_pts, seed=seed, variant="J", return_half=True)
        q = synth.rrt_queries(n_q, half, seed=seed + 1)
        cases.append((torch.from_numpy(pts).to(dev), torch.from_numpy(q).to(dev)))
    libs = [("default", os.path.join(ROOT, "pointcloudtraj_b200", "libpcindex.so"))] + [(os.path.basename(p)[4:-3], p) for p in sorted(glob.glob(os.path.join(ROOT, "build", "variants", "lib_*.so")))]
    vp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    calls = (("range", None), ("sorted0", 0), ("sorted64", 64))
    print(f"{'variant':24s} " + " ".join(f"{w + ' ' + c:>14s}" for w in ("c1", "1M/50k") for c, _ in calls) + "  (ms) same")
    ref = None
    for _ in range(a.rounds):
        for name, path in libs:
            _lib._lib = None
            _lib.LIB_PATH = path
            L = _lib.load()
            row, outs = [], []
            for t_pts, t_q in cases:
                h = C.c_void_p()
                assert L.pc_index_create(C.byref(h), 0, t_pts.shape[0], C.c_void_p(stream)) == 0
                assert L.pc_index_build(h, vp(t_pts), t_pts.shape[0], 3, 1) == 0
                m = t_q.shape[0]
                t_r = torch.ones(1, dtype=torch.float64, device=dev)
                for _, max_nn in calls:
                    def run(off, idx, d2, cap):
                        if max_nn is None:
                            return L.pc_range_batch(h, vp(t_q), m, 3, 1, vp(t_r), 1, vp(off), vp(idx), cap)
                        return L.pc_range_sorted_batch(h, vp(t_q), m, 3, 1, vp(t_r), 1, max_nn, vp(off), vp(idx), vp(d2), cap)
                    t_off = torch.empty(m + 1, dtype=torch.int64, device=dev)
                    assert run(t_off, None, None, 0) == 0
                    torch.cuda.synchronize()
                    total = int(t_off[-1].item())
                    t_lst = torch.empty(total, dtype=torch.int32, device=dev)
                    t_d2 = torch.empty(total, dtype=torch.float32, device=dev) if max_nn is not None else None
                    ms = []
                    for _ in range(9):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        assert run(t_off, t_lst, t_d2, total) == 0
                        e1.record()
                        torch.cuda.synchronize()
                        ms.append(e0.elapsed_time(e1))
                    row.append(float(np.median(ms[2:])))
                    outs.append([t.cpu().numpy().copy() for t in (t_off, t_lst, t_d2) if t is not None])
                L.pc_index_destroy(h)
            if ref is None:
                ref = outs
            same = all(len(x) == len(y) and all(np.array_equal(u.view(np.uint8), v.view(np.uint8)) for u, v in zip(x, y)) for x, y in zip(ref, outs))
            print(f"{name:24s} " + " ".join(f"{v:14.3f}" for v in row) + f"  {same}", flush=True)


if __name__ == "__main__":
    main()
