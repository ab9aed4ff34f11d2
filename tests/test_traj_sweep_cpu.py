"""CPU checks of the trajectory-sweep oracle (tests/traj_sweep_brute.py) against dense sampling, the closed-form first root on
straight segments and hand-built starts in contact; its motion rule; and pc_trajectory_sweep_batch's NULL-handle refusal."""
import ctypes as C

import numpy as np
import pytest

from pointcloudtraj_b200 import _lib as L

import traj_sweep_brute as TB


def _curve(rng, n, scale=2.0):
    P = np.cumsum(rng.normal(size=(n + 1, 3)) * scale / max(n, 1), 0)
    return P


@pytest.mark.parametrize("n", range(1, 13))
def test_oracle_vs_dense_sampling(n):
    rng = np.random.default_rng(100 + n)
    for trial in range(6):
        P = _curve(rng, n)
        u = np.linspace(0.0, 1.0, 20001)
        curve = np.array([TB.evaluate(P, x) for x in u[::50]])
        pts = curve[rng.integers(0, len(curve), 40)] + rng.normal(size=(40, 3)) * 0.3
        rho = 0.2
        cloud = TB.CloudBoxes(pts.astype(np.float32))
        pw = cloud.p
        res = TB.first_contact_segment(P, 1.0, 0.0, 1.0, cloud, rho)
        dense = np.array([TB.evaluate(P, x) for x in u])
        d = np.sqrt(((dense[:, None, :] - pw[None, :, :]) ** 2).sum(-1)).min(1)
        hit = np.nonzero(d <= rho)[0]
        if res is None:
            assert len(hit) == 0 or d.min() > rho - 1e-9
            continue
        sigma, i = res
        # nothing earlier (up to the sampling's own resolution), and the point touches there
        assert len(hit) == 0 or sigma <= u[hit[0]] + 1e-12
        early = u < sigma - 1e-9
        assert (d[early] > rho - 1e-9).all()
        p = cloud.p[np.nonzero(cloud.idx == i)[0][0]]
        assert np.linalg.norm(TB.evaluate(P, sigma) - p) <= rho + 1e-9


def test_oracle_straight_segments_closed_form():
    rng = np.random.default_rng(7)
    for trial in range(200):
        a, b = rng.uniform(-3, 3, 3), rng.uniform(-3, 3, 3)
        n = int(rng.integers(1, 13))
        P = a + np.linspace(0, 1, n + 1)[:, None] * (b - a)          # a straight segment at any order (uniform parameter)
        p = a + rng.uniform(0, 1) * (b - a) + rng.normal(size=3) * 0.5
        rho = float(rng.uniform(0.05, 1.0))
        cloud = TB.CloudBoxes(p[None].astype(np.float32))
        pw = cloud.p[0]
        D, W = b - a, pw - a
        qa, qb, qc = D @ D, -2 * (W @ D), W @ W - rho * rho
        disc = qb * qb - 4 * qa * qc
        if qc <= 0:
            want = 0.0
        elif disc < 0:
            want = None
        else:
            t0 = (-qb - np.sqrt(disc)) / (2 * qa)
            want = t0 if 0 <= t0 <= 1 else None
        res = TB.first_contact_segment(P, 1.0, 0.0, 1.0, cloud, rho)
        if want is None:
            assert res is None or abs(np.sqrt(disc)) < 1e-6
        else:
            assert res is not None and abs(res[0] - want) <= 1e-10


def test_oracle_start_inside_contact_and_motion_part():
    rng = np.random.default_rng(3)
    P = _curve(rng, 5)
    T = 2.0
    for sa in (0.0, 0.3, 1.1, 2.0):
        c = TB.evaluate(P, sa / T)
        cloud = TB.CloudBoxes((c + np.array([0.05, 0.0, 0.0]))[None].astype(np.float32))
        res = TB.first_contact_segment(P, T, sa, T, cloud, 0.1)
        assert res is not None and res[0] == sa


def test_motion_rule():
    T = np.array([0.5, 0.75, 1.0])
    assert TB.motion(0, 3, -1.0, T, 2.0) == [(0, 0.0, 0.5), (1, 0.0, 0.75), (2, 0.0, 0.75)]
    assert TB.motion(0, 3, 0.5, T, 0.25) == [(0, 0.5, 0.5), (1, 0.0, 0.25)]
    assert TB.motion(0, 3, np.nextafter(0.5, 1), T, 0.1)[0][0] == 1
    assert TB.motion(0, 3, 5.0, T, 1.0) == []                     # past the end
    assert TB.motion(0, 3, 2.25, T, 1.0) == [(2, 1.0, 1.0)]       # exactly the end
    assert TB.motion(0, 3, 0.0, T, 0.0) == [(0, 0.0, 0.0)]
    assert TB.motion(0, 3, 0.0, T, -0.5) == []
    assert TB.motion(0, 3, 0.0, T, 1.25) == [(0, 0.0, 0.5), (1, 0.0, 0.75), (2, 0.0, 0.0)]   # a boundary
    assert TB.motion(0, 0, 0.0, T, 1.0) == []


def test_null_handle_is_rejected():
    lib = L.load()
    tr = L.PcTraj(0, 1, 0.0)
    order = (C.c_int32 * 1)(1)
    Ts = (C.c_double * 1)(1.0)
    off = (C.c_int64 * 1)(0)
    coef = (C.c_double * 6)()
    out = (C.c_int32 * 1)(), (C.c_double * 1)(), (C.c_int32 * 1)()
    rc = lib.pc_trajectory_sweep_batch(None, C.byref(tr), 1, order, Ts, off, 1, coef, 6, L.PC_HOST, 1.0, 0.5, 1e-3, *out)
    assert rc == L.PC_EINVAL
