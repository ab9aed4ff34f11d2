"""Counts of the 64-query packet walk on the bench workload, emulated on the CPU (scripts/packet_emu.cpp): node visits, leaf scans
and fp64 re-checks per packet, one fp64 site per point (the old leaf scan) against one per query slot (pc_exact_leaf), for a walk
from the root and from entry frontiers of at most K subtrees.

    python scripts/packet_emu.py [--queries 10000000] [--stride 1] [--entries 0 1 4 8] [--out profiles/r3_packet_emu.txt]

The workload is bench.py's: the 1 M-point C2 map, one step's uniform in-box samples (seed 1000), the queries outside the sensing
range (answered by radiusSearch's early-out, never searched) dropped, radius bound max_radius + search_margin = 1.75 m.  Queries are
ordered by the top 24 bits of their Hilbert key (the radix-sort ordering pass; bench batches take the cell binning, which groups them
alike).  --stride k walks every k-th packet only.  Every figure is a CPU count, not a GPU measurement."""
import argparse
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=10_000_000)
    ap.add_argument("--stride", type=int, default=1)
    ap.add_argument("--entries", type=int, nargs="+", default=[0, 1, 4, 8], help="0 = from the root")
    ap.add_argument("--dil", type=float, default=1.75, help="dilation of a packet's box for the entry frontier (m)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from pointcloudtraj_b200 import synth
    search_margin, max_radius, sample_range, start = 0.25, 1.5, 30.0, np.array([0.0, 0.0, 2.0])
    pts, half = synth.forest_cloud(1_000_000, seed=1, variant="J", return_half=True)
    q = synth.rrt_queries(args.queries, half, seed=1000)
    d = np.sqrt(((q.astype(np.float32).astype(np.float64) - start) ** 2).sum(axis=1))
    q = q[~(d > sample_range + max_radius)]
    lines = [f"# scripts/packet_emu.py --queries {args.queries} --stride {args.stride} --dil {args.dil}: "
             f"{len(q)} searched queries of {args.queries} (the rest take the sensing-range early-out)"]
    with tempfile.TemporaryDirectory() as tmp:
        exe, fp, fq = os.path.join(tmp, "packet_emu"), os.path.join(tmp, "p.bin"), os.path.join(tmp, "q.bin")
        subprocess.run(["g++", "-std=c++14", "-O2", "-ffp-contract=off", "-o", exe, os.path.join(ROOT, "scripts", "packet_emu.cpp")], check=True)
        np.ascontiguousarray(pts[:, :3], np.float32).tofile(fp)
        np.ascontiguousarray(q, np.float32).tofile(fq)
        for k in args.entries:
            r = subprocess.run([exe, fp, fq, str(search_margin + max_radius), f"K={k}", f"dil={args.dil}", f"stride={args.stride}"],
                               capture_output=True, text=True, check=True)
            lines.append(r.stdout.strip())
            print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
