"""CPU check of the leaf scan's fp64 re-check rule (pc_exact_leaf in query_kernels.cuh: only the points within the fp32 margin of
the leaf's minimum are re-evaluated) through the packet-walk emulator scripts/packet_emu.cpp: on a tie-heavy lattice forest the
walk with the new rule agrees, leaf by leaf, with the walk that re-checks every point under the threshold (the emulator exits
otherwise), and every result equals an fp64 brute force; bounded and unbounded, and from entry frontiers."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_exact_leaf_rule_matches_brute_force(tmp_path):
    import numpy as np
    from pointcloudtraj_b200 import synth
    exe = str(tmp_path / "packet_emu")
    subprocess.run(["g++", "-std=c++14", "-O2", "-ffp-contract=off", "-o", exe, os.path.join(ROOT, "scripts", "packet_emu.cpp")],
                   check=True, capture_output=True)
    pts, half = synth.forest_cloud(20_000, seed=6, variant="L", return_half=True)
    q = synth.rrt_queries(2000, half, seed=3)
    q[::2] = np.round(q[::2] / 0.05) * 0.05
    fp, fq = str(tmp_path / "p.bin"), str(tmp_path / "q.bin")
    np.ascontiguousarray(pts[:, :3], np.float32).tofile(fp)
    np.ascontiguousarray(q, np.float32).tofile(fq)
    for bound, extra in (("1.75", []), ("1.75", ["K=4"]), ("0", [])):
        r = subprocess.run([exe, fp, fq, bound, "check"] + extra, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "mismatches=0" in r.stdout, (bound, extra, r.stdout, r.stderr)
