"""Drop-in check of include/pc_kdtree_compat.h: the SAME C client (tests/c/kd_client.c, written against the reference's
kd_* API) is built once on the unmodified reference library and once on libpcindex via the kd_* -> pckd_* renames;
both runs must produce the same output on the same input."""
import os
import struct
import subprocess

import numpy as np
import pytest

import oracle
from pointcloudtraj_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(tmp, name, extra):
    exe = os.path.join(tmp, name)
    cmd = ["gcc", "-O2", "-o", exe, os.path.join(ROOT, "tests", "c", "kd_client.c")] + extra
    subprocess.run(cmd, check=True, capture_output=True)
    return exe


def _read(path, m, nr):
    raw = open(path, "rb").read()
    nn = np.frombuffer(raw, np.int64, m, 0)
    pos = np.frombuffer(raw, np.float64, 3 * m, 8 * m).reshape(m, 3)
    cnt = np.frombuffer(raw, np.int64, nr, 32 * m)
    items = np.frombuffer(raw, np.int64, int(cnt.sum()), 32 * m + 8 * nr)
    return nn, pos, cnt, items


@pytest.mark.skipif(not oracle.have_reference(), reason="needs the upstream pointcloudTraj kd-tree compiled into oracle/_ref (make -C oracle REF=<pointcloudTraj checkout>)")
def test_same_client_two_backends(tmp_path):
    tmp = str(tmp_path)
    pts, half = synth.forest_cloud(40_000, seed=8, variant="J", return_half=True)
    q = synth.rrt_queries(1500, half, seed=9)
    nr, rng = 150, 0.75
    with open(os.path.join(tmp, "in.bin"), "wb") as f:
        f.write(struct.pack("<qqqd", len(pts), len(q), nr, rng))
        f.write(pts.tobytes())
        f.write(q.tobytes())
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    lib_dir = os.path.join(ROOT, "pointcloudtraj_b200")
    ref_exe = _build(tmp, "client_ref", ["-L", ref_dir, "-lkdtree_ref", f"-Wl,-rpath,{ref_dir}", "-lm"])
    gpu_exe = _build(tmp, "client_gpu", ["-DUSE_PCINDEX", "-I", os.path.join(ROOT, "include"), "-L", lib_dir, "-lpcindex",
                                         f"-Wl,-rpath,{lib_dir}"])
    for exe, out in ((ref_exe, "ref.bin"), (gpu_exe, "gpu.bin")):
        p = subprocess.run([exe, os.path.join(tmp, "in.bin"), os.path.join(tmp, out)], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, (exe, p.returncode, p.stderr)
    a = _read(os.path.join(tmp, "ref.bin"), len(q), nr)
    b = _read(os.path.join(tmp, "gpu.bin"), len(q), nr)
    assert (a[0] == b[0]).all()            # same nearest point (data pointer) for every query: tie-free cloud
    assert (a[1] == b[1]).all()            # same coordinates handed back by kd_res_item
    assert (a[2] == b[2]).all() and (a[3] == b[3]).all()   # same range sets
    assert a[2].sum() > 1000


def test_corridor_wrapper_matches_radius_search_oracle(tmp_path):
    """include/pc_corridor.hpp (C++ mirror of safeRegionRrtStar's cloud-facing members) against the restated radiusSearch."""
    tmp = str(tmp_path)
    pts, half = synth.forest_cloud(30_000, seed=3, variant="J", return_half=True)
    rng = np.random.default_rng(4)
    q = np.stack([rng.uniform(-1.6 * half, 1.6 * half, 800), rng.uniform(-1.6 * half, 1.6 * half, 800), rng.uniform(0.6, 4.0, 800)], 1)
    prm = (0.6, 0.25, 1.5, 14.0)
    start = (1.0, -1.0, 2.0)
    pts4 = np.concatenate([pts, np.zeros((len(pts), 1), np.float32)], 1)
    with open(os.path.join(tmp, "in.bin"), "wb") as f:
        f.write(struct.pack("<qq4d3d", len(pts), len(q), *prm, *start))
        f.write(pts4.tobytes())
        f.write(q.astype(np.float64).tobytes())
    lib_dir = os.path.join(ROOT, "pointcloudtraj_b200")
    exe = os.path.join(tmp, "corridor_client")
    subprocess.run(["g++", "-std=c++14", "-O2", "-o", exe, os.path.join(ROOT, "tests", "c", "corridor_client.cpp"),
                    "-I", os.path.join(ROOT, "include"), "-L", lib_dir, "-lpcindex", f"-Wl,-rpath,{lib_dir}"], check=True, capture_output=True)
    p = subprocess.run([exe, os.path.join(tmp, "in.bin"), os.path.join(tmp, "out.bin")], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, (p.returncode, p.stderr)
    raw = open(os.path.join(tmp, "out.bin"), "rb").read()
    m = len(q)
    r_single = np.frombuffer(raw, np.float64, m, 0)
    r_batch = np.frombuffer(raw, np.float32, m, 8 * m)
    col = np.frombuffer(raw, np.uint8, m, 12 * m)
    ko = oracle.KdOracle().build(pts, np.random.default_rng(1).permutation(len(pts)))
    P = oracle.RadiusParams.make(prm[1], prm[2], prm[3], start)
    ref = np.array([ko.radius_search(P, q[k])[0] for k in range(m)])          # double points, as the planner passes them
    assert (r_single == ref.astype(np.float32).astype(np.float64)).all()
    ref_b, _ = ko.radius_batch(P, q.astype(np.float32))                       # float32 points, as the batch ABI takes them
    assert (r_batch == ref_b.astype(np.float32)).all()
    assert (col.astype(bool) == (ref_b < 0)).all()
    assert (ref == prm[2] - prm[1]).any() and (ref < 0).any() and (ref == prm[2]).any()
    # the ground-truth collision arbiter (status_inspector.cpp:33-46) against the oracle's exact nearest distances:
    # sqrt (float32, as the reference computes it from PCL's float distances) of d2 < col_rad, first such position
    first_col, = struct.unpack_from("<q", raw, 13 * m)
    nd = np.frombuffer(raw, np.float32, m, 13 * m + 8)
    _, od2 = ko.nearest(q.astype(np.float32))
    od = np.sqrt(od2.astype(np.float32))
    assert (nd == od).all()
    hits = np.nonzero(od.astype(np.float64) < 0.3)[0]
    assert first_col == (hits[0] if len(hits) else -1) and len(hits) > 0
