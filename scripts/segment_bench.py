#!/usr/bin/env python
"""pc_segment_nearest_batch sweep: device-resident batches timed with CUDA events (median of repeated calls after warm-up).

    python scripts/segment_bench.py [--m 1000000] [--bound 0.5] [--h 0.25] [--order-sizes ...] [--out FILE]

Workloads: C2 = the bench map (synth.forest_cloud(1_000_000, variant="J")) and C1 = synth.forest_cloud(200_000, variant="J"),
--m segments each, starts uniform in the cloud's bounding box, random directions, lengths 0, 0.1, 1 and 10 m.
For every length and bound (unbounded, --bound m) it times PC_QUERY_UNSORTED, PC_QUERY_SORTED and PC_QUERY_AUTO; all three
must return the same bits (ok=True).  Comparison with the same guarantee: pc_nearest_batch (AUTO) on points
sampled every h along each segment (ceil(len / h) + 1 per segment, both ends included), whose clearance check then needs the
radius inflated by h / 2.  A last section times SORTED against UNSORTED on C2 from 1 k to 1 M segments (the crossover of
PC_QUERY_AUTO).  Each line: median ms per call, [min, max] over the timed calls, segments/s of the median.  The card's name,
power limit and max / current SM clock are printed first.
"""
import argparse
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def segments(pts, m, length, seed):
    rng = np.random.default_rng(seed)
    lo, hi = pts.min(0).astype(np.float64), pts.max(0).astype(np.float64)
    a = rng.uniform(lo, hi, (m, 3))
    d = rng.normal(size=(m, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return a.astype(np.float32), (a + d * length).astype(np.float32)


def samples(a, b, h):
    """points every h along each segment, both ends included (float32, (sum, 3))"""
    L = np.linalg.norm(b.astype(np.float64) - a.astype(np.float64), axis=1)
    k = np.ceil(L / h).astype(np.int64) + 1
    seg = np.repeat(np.arange(len(a)), k)
    first = np.repeat(np.cumsum(k) - k, k)
    t = (np.arange(k.sum()) - first) / np.maximum(k[seg] - 1, 1)
    return (a[seg] + t[:, None] * (b[seg] - a[seg]).astype(np.float64)).astype(np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--m", type=int, default=1_000_000)
    ap.add_argument("--lengths", default="0,0.1,1,10")
    ap.add_argument("--bound", type=float, default=0.5)
    ap.add_argument("--h", type=float, default=0.25)
    ap.add_argument("--order-sizes", default="1000,8000,32000,100000,300000,1000000")
    ap.add_argument("--order-lengths", default="0.1,1,10")
    ap.add_argument("--skip-sweep", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("segment_bench.py needs a CUDA device")
    from pointcloudtraj_b200 import PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED, PointCloudIndex, synth

    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    def smi():
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name(0)

    emit(f"# GPU: {smi()} (name, power limit, max SM clock, current SM clock)")
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
        return f"{name:52s} m={m:>8d}  {med:9.4f} ms  [{lo:.4f}, {hi:.4f}]  {m / (med * 1e-3):.3e} seg/s"

    def rname(r):
        return f"r={r}" if r is not None else "unbounded"

    names = {PC_QUERY_UNSORTED: "UNSORTED", PC_QUERY_SORTED: "SORTED", PC_QUERY_AUTO: "AUTO"}

    def index_of(pts):
        ix = PointCloudIndex(max_points=len(pts), device=0, stream=st.cuda_stream)
        ix.build(pts)
        ix.sync()
        return ix

    c2 = synth.forest_cloud(1_000_000, variant="J")
    if not a.skip_sweep:
        for cname, pts in (("C2", c2), ("C1", synth.forest_cloud(200_000, variant="J"))):
            ix = index_of(pts)
            lo, hi = pts.min(0), pts.max(0)
            emit(f"## {cname}: forest_cloud({len(pts)}, variant='J'), box {lo.round(2).tolist()} .. {hi.round(2).tolist()}; "
                 f"{a.m} segments, starts uniform in the box")
            for length in [float(s) for s in a.lengths.split(",")]:
                sa, sb = segments(pts, a.m, length, seed=1)
                da, db = torch.from_numpy(sa).cuda(), torch.from_numpy(sb).cuda()
                smp = torch.from_numpy(samples(sa, sb, a.h)).cuda()
                for r in (None, a.bound):
                    ref = None
                    ok = True
                    for fl in (PC_QUERY_UNSORTED, PC_QUERY_SORTED, PC_QUERY_AUTO):
                        emit(fmt(f"len={length:<5g} {rname(r):9s} {names[fl]}", a.m, timed(lambda: ix.segment_nearest(da, db, r, fl), a.m)))
                        gi, gd = ix.segment_nearest(da, db, r, fl)
                        got = (gi.cpu().numpy(), gd.cpu().numpy().view(np.uint32))
                        if ref is None:
                            ref = got
                        ok = ok and (got[0] == ref[0]).all() and (got[1] == ref[1]).all()
                    hit = int((ref[0] >= 0).sum())
                    emit(f"len={length:<5g} {rname(r):9s} ok={ok}  rows with a point: {hit}")
                emit(fmt(f"len={length:<5g} sampled h={a.h} nearest ({smp.shape[0]} samples)", a.m,
                         timed(lambda: ix.nearest(smp), a.m)))
                del da, db, smp
                torch.cuda.empty_cache()
            ix.close()

    # the ordering crossover on the bench map
    ix = index_of(c2)
    sizes = [int(s) for s in a.order_sizes.split(",")]
    emit("## ordering crossover on C2: UNSORTED ms / SORTED ms / AUTO ms (faster forced path)")
    for length in [float(s) for s in a.order_lengths.split(",")]:
        sa, sb = segments(c2, max(sizes), length, seed=2)
        for r in (None, a.bound):
            for m in sizes:
                da, db = torch.from_numpy(sa[:m]).cuda(), torch.from_numpy(sb[:m]).cuda()
                t = {fl: timed(lambda: ix.segment_nearest(da, db, r, fl), m)[0] for fl in (PC_QUERY_UNSORTED, PC_QUERY_SORTED, PC_QUERY_AUTO)}
                fast = "SORTED" if t[PC_QUERY_SORTED] < t[PC_QUERY_UNSORTED] else "UNSORTED"
                emit(f"len={length:<5g} {rname(r):9s} m={m:>8d}  {t[PC_QUERY_UNSORTED]:9.4f} {t[PC_QUERY_SORTED]:9.4f} {t[PC_QUERY_AUTO]:9.4f}  faster={fast}")
    ix.close()
    emit(f"# GPU after the run: {smi()}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
