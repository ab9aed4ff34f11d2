"""The numpy oracle of pc_trajectory_nearest_batch (tests/traj_nearest_brute.py) against dense sampling, closed forms and the
first-contact oracle of tests/traj_sweep_brute.py.  No GPU needed."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from pointcloudtraj_b200 import synth

import traj_nearest_brute as NB
import traj_sweep_brute as TB


def _one(P_list, T_list):
    order = np.array([len(P) - 1 for P in P_list], np.int32)
    T = np.array(T_list, np.float64)
    off = np.zeros(len(P_list) + 1, np.int64)
    off[1:] = np.cumsum(3 * (order + 1))
    coef = np.concatenate([(np.asarray(P, np.float64) / T[i]).T.ravel() for i, P in enumerate(P_list)])
    return dict(traj_first_seg=np.array([0, len(P_list)], np.int32), seg_order=order, seg_T=T, seg_coef_off=off, coef=coef)


@pytest.fixture(scope="module")
def small_forest():
    pts, half = synth.forest_cloud(20_000, seed=4, variant="J", return_half=True)
    return pts, half, NB.NearestOracle(pts)


def test_dense_sampling(small_forest):
    pts, half, orc = small_forest
    tr = synth.bezier_trajectories(40, half * 0.9, seed=5, order_range=(1, 12))
    tree = cKDTree(orc.cloud.p)
    u = np.linspace(0.0, 1.0, 4001)
    for t in range(40):
        lo, hi = orc.bracket(tr, t, 0.0, 2.0)
        assert np.isfinite(lo) and lo <= hi and hi - lo <= 1e-7, (t, lo, hi)
        m = np.inf
        for Q in NB._parts(tr, t, 0.0, 2.0):
            X = np.stack([TB.evaluate(Q, v) for v in u])
            m = min(m, float(tree.query(X)[0].min()))
        assert lo <= m + 1e-12 and m - hi <= 1e-3, (t, lo, hi, m)


def test_straight_segments_closed_form():
    rng = np.random.default_rng(3)
    a = rng.uniform(-5, 5, (30, 3))
    b = a + rng.normal(size=(30, 3)) * 3
    pts = rng.uniform(-6, 6, (3000, 3)).astype(np.float32)
    P = pts.astype(np.float64)
    orc = NB.NearestOracle(pts)
    for k in range(30):
        for order in (1, 4):
            ctrl = a[k] + np.linspace(0, 1, order + 1)[:, None] * (b[k] - a[k])      # a straight segment of any order
            lo, hi = orc.bracket(_one([ctrl], [1.5]), 0, 0.0, 10.0)
            d = b[k] - a[k]
            t = np.clip(((P - a[k]) @ d) / (d @ d), 0.0, 1.0)
            exact = np.linalg.norm(P - (a[k] + t[:, None] * d), axis=1).min()
            assert lo <= exact + 1e-12 <= hi + 2e-12 and hi - lo <= 1e-7, (k, order, lo, hi, exact)


@pytest.mark.parametrize("a", [0.3, 0.45, 1.2, 2.0])
def test_parabola_vertex(a):
    """C(v) = (x, x^2, 0), x = 2v - 1 in [-1, 1]: from (0, a, 0) the vertex is nearest for a <= 1/2 (distance a), then
    x^2 = a - 1/2 (distance sqrt(a - 1/4)) up to a = 3/2, beyond that the ends (distance sqrt(1 + (1 - a)^2))."""
    ctrl = np.array([[-1.0, 1.0, 0.0], [0.0, -1.0, 0.0], [1.0, 1.0, 0.0]])
    p = np.array([[0.0, a, 0.0]], np.float32)
    af = float(p[0, 1])
    exact = af if af <= 0.5 else np.sqrt(af - 0.25) if af <= 1.5 else np.sqrt(1 + (1 - af) ** 2)
    lo, hi = NB.NearestOracle(p).bracket(_one([ctrl], [1.0]), 0, 0.0, 10.0)
    assert lo <= exact <= hi and hi - lo <= 1e-7, (lo, hi, exact)


def test_first_contact_at_the_bracket(small_forest):
    pts, half, orc = small_forest
    tr = synth.bezier_trajectories(25, half * 0.9, seed=9, order_range=(1, 12))
    for t in range(25):
        lo, hi = orc.bracket(tr, t, 0.3, 2.0)
        assert TB.first_contact(tr, t, 0.3, orc.cloud, hi * (1 + 1e-9) + 1e-9, 2.0) is not None, (t, hi)
        if lo > 1e-6:
            assert TB.first_contact(tr, t, 0.3, orc.cloud, lo * (1 - 1e-6), 2.0) is None, (t, lo)


def test_empty_motion_and_empty_cloud():
    ctrl = np.array([[0.0, 0.0, 1.0], [1.0, 0.0, 1.0]])
    tr = _one([ctrl], [1.0])
    assert NB.NearestOracle(np.array([[0, 0, 0]], np.float32)).bracket(tr, 0, 5.0, 2.0) == (np.inf, np.inf)
    assert NB.NearestOracle(np.full((4, 3), np.nan, np.float32)).bracket(tr, 0, 0.0, 2.0) == (np.inf, np.inf)
    lo, hi = NB.NearestOracle(np.array([[0.5, 0, 1]], np.float32)).bracket(tr, 0, 0.0, 2.0)
    assert lo == 0.0 and hi <= 1e-6                      # near 0 the bracket is as wide as fp64 resolves |C - p|^2
