"""pc_trajectory_nearest_batch on the GPU: every answer is checked against the numpy bracket [lo, hi] of D* (tests/
traj_nearest_brute.py) for the contract's three rules -- a witness position and point at most d apart (re-evaluated in fp64
here), nothing closer than d - tol, and the max_range bound -- with a slack of 1e-9 far below every tol used; and against
pc_trajectory_sweep_batch, pc_clearance_batch and pc_segment_nearest_batch on the same inputs."""
import ctypes as C

import numpy as np
import pytest

from pointcloudtraj_b200 import PointCloudIndex, PcRadiusParams, synth
from pointcloudtraj_b200 import _lib as L

import traj_nearest_brute as NB
import traj_sweep_brute as TB

pytestmark = pytest.mark.gpu
SLACK = 1e-9


def _vp(a):
    return C.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)


def _traj_records(tr, t_now):
    first = tr["traj_first_seg"]
    n = len(first) - 1
    rec = np.zeros(max(n, 1), dtype=np.dtype([("first_seg", "<i4"), ("num_seg", "<i4"), ("t_now", "<f8")]))
    rec["first_seg"][:n], rec["num_seg"][:n], rec["t_now"][:n] = first[:-1], np.diff(first), t_now
    return rec


def nearest(ix, tr, t_now, max_range, tol, horizon, space=L.PC_HOST):
    """The C call in either space (PC_DEVICE: every array a CUDA tensor), outputs pre-filled with a sentinel."""
    n = len(tr["traj_first_seg"]) - 1
    arrays = [_traj_records(tr, t_now).view(np.uint8), np.ascontiguousarray(tr["seg_order"], np.int32),
              np.ascontiguousarray(tr["seg_T"], np.float64), np.ascontiguousarray(tr["seg_coef_off"], np.int64),
              np.ascontiguousarray(tr["coef"], np.float64)]
    outs = [np.full(n, -7, np.int32), np.full(n, -7.0), np.full(n, -7, np.int32), np.full(n, -7.0)]
    if space == L.PC_DEVICE:
        import torch
        arrays = [torch.from_numpy(a).cuda() for a in arrays]
        outs = [torch.from_numpy(a).cuda() for a in outs]
        torch.cuda.synchronize()
    rc = ix._L.pc_trajectory_nearest_batch(ix._h, _vp(arrays[0]), n, _vp(arrays[1]), _vp(arrays[2]), _vp(arrays[3]),
                                           len(tr["seg_order"]), _vp(arrays[4]), len(tr["coef"]), space, float(horizon),
                                           float(max_range), float(tol), *[_vp(o) for o in outs])
    assert rc == L.PC_OK, ix._L.pc_last_error(ix._h)
    if space == L.PC_DEVICE:
        ix.sync()
        outs = [o.cpu().numpy() for o in outs]
    return outs


def brackets(orc, tr, t_now, horizon, which=None):
    n = len(tr["traj_first_seg"]) - 1
    t_now = np.broadcast_to(np.asarray(t_now, np.float64), (n,))
    return {t: orc.bracket(tr, t, t_now[t], horizon) for t in (range(n) if which is None else which)}


def check_rules(tr, t_now, orc, br, max_range, tol, horizon, seg, s, idx, dist):
    """The three rules for the trajectories of the brackets br; returns the number of rows with a witness."""
    n = len(tr["traj_first_seg"]) - 1
    t_now = np.broadcast_to(np.asarray(t_now, np.float64), (n,))
    found = 0
    for t, (lo, hi) in br.items():
        if seg[t] < 0:
            assert idx[t] == -1 and s[t] == np.inf and dist[t] == np.inf, (t, seg[t], s[t], idx[t], dist[t])
            assert (hi >= max_range - SLACK) if max_range >= 0 else hi == np.inf, f"trajectory {t}: no witness, D* <= {hi}"
            continue
        found += 1
        mot = TB.motion(int(tr["traj_first_seg"][t]), int(tr["traj_first_seg"][t + 1] - tr["traj_first_seg"][t]), float(t_now[t]),
                        tr["seg_T"], horizon)
        sg, sa, sb = mot[[m[0] for m in mot].index(int(seg[t]))]
        T = float(tr["seg_T"][sg])
        assert sa <= s[t] <= sb + SLACK * T, (t, s[t], sa, sb)
        P = TB.polygon(tr["coef"], tr["seg_coef_off"], tr["seg_order"], tr["seg_T"], sg)
        k = np.nonzero(orc.cloud.idx == idx[t])[0]
        assert len(k) == 1, f"trajectory {t}: witness {idx[t]} is not a finite cloud point"
        e = np.linalg.norm(TB.evaluate(P, s[t] / T) - orc.cloud.p[k[0]])
        assert e <= dist[t] + SLACK, f"trajectory {t}: witness at {e}, d = {dist[t]}"                         # rule 1
        assert lo >= dist[t] - tol - SLACK, f"trajectory {t}: D* >= {lo} but d - tol = {dist[t] - tol}"        # rule 2
        assert max_range < 0 or dist[t] <= max_range + tol + SLACK, (t, dist[t], max_range)                  # rule 3
    return found


def _mixed_t_now(n, rng):
    t = np.zeros(n)
    sel = rng.random(n) < 0.3
    t[sel] = rng.uniform(-1.0, 4.0, int(sel.sum()))
    return t


@pytest.fixture(scope="module")
def forest():
    pts, half = synth.forest_cloud(200_000, seed=11, variant="J", return_half=True)
    ix = PointCloudIndex(max_points=len(pts), device=0)
    ix.build(pts)
    orc = NB.NearestOracle(pts)
    tr = synth.bezier_trajectories(1000, half * 0.9, seed=21, order_range=(1, 12))
    t_now = _mixed_t_now(1000, np.random.default_rng(5))
    yield pts, half, ix, orc, tr, t_now, brackets(orc, tr, t_now, 2.0)
    ix.close()


@pytest.mark.parametrize("tol", [1e-3, 1e-5])
@pytest.mark.parametrize("max_range", [-1.0, 0.0, 0.3, 2.0])
def test_forest_rules_both_spaces(forest, max_range, tol):
    pts, half, ix, orc, tr, t_now, br = forest
    host = nearest(ix, tr, t_now, max_range, tol, 2.0)
    dev = nearest(ix, tr, t_now, max_range, tol, 2.0, L.PC_DEVICE)
    again = nearest(ix, tr, t_now, max_range, tol, 2.0)
    for a, b, c in zip(host, dev, again):
        assert a.tobytes() == b.tobytes() == c.tobytes()
    n = check_rules(tr, t_now, orc, br, max_range, tol, 2.0, *host)
    assert max_range == 0.0 or n > 100


def test_relation_with_trajectory_sweep(forest):
    """d <= r: the sweep at r reports a contact; d - tol > r + the sweep's tol: it reports none."""
    pts, half, ix, orc, tr, t_now, br = forest
    r, stol, tol = 0.5, 1e-3, 1e-4
    seg, s, idx, dist = nearest(ix, tr, t_now, -1.0, tol, 2.0)
    n = len(seg)
    rec = _traj_records(tr, t_now)
    so, sT = np.ascontiguousarray(tr["seg_order"], np.int32), np.ascontiguousarray(tr["seg_T"], np.float64)
    sc, cf = np.ascontiguousarray(tr["seg_coef_off"], np.int64), np.ascontiguousarray(tr["coef"], np.float64)
    wseg, ws, widx = np.zeros(n, np.int32), np.zeros(n), np.zeros(n, np.int32)
    assert ix._L.pc_trajectory_sweep_batch(ix._h, _vp(rec), n, _vp(so), _vp(sT), _vp(sc), len(so), _vp(cf), len(cf), L.PC_HOST,
                                           2.0, r, stol, _vp(wseg), _vp(ws), _vp(widx)) == L.PC_OK
    assert (wseg[dist <= r] >= 0).all()
    assert (wseg[dist - tol > r + stol] == -1).all()
    assert ((seg >= 0) == np.isfinite(dist)).all() and (np.isinf(dist) <= (wseg == -1)).all()
    assert (dist <= r).sum() > 20 and (dist - tol > r + stol).sum() > 20


def test_relation_with_clearance(forest):
    """pc_clearance_batch's sampled radii can never undercut the certificate: min_radius + search_margin >= d - tol - c, with c
    the float32 cast of the sample positions and the float32 rounding of min_radius."""
    pts, half, ix, orc, tr, t_now, br = forest
    tol, margin = 1e-4, 0.25
    seg, s, idx, dist = nearest(ix, tr, 0.0, -1.0, tol, 2.0)
    params = PcRadiusParams.make(margin, 1e3, -1.0, (0.0, 0.0, 0.0))
    fh, mr, ns = ix.clearance(tr["traj_first_seg"], tr["seg_order"], tr["seg_T"], tr["seg_coef_off"], tr["coef"], params,
                              dt=0.02, horizon=2.0)
    first = tr["traj_first_seg"]
    checked = 0
    for t in range(len(first) - 1):
        if ns[t] == 0 or seg[t] < 0:
            continue
        xmax = max(np.abs(TB.polygon(tr["coef"], tr["seg_coef_off"], tr["seg_order"], tr["seg_T"], sg)).max()
                   for sg in range(first[t], first[t + 1]))
        c = xmax * 2.0 ** -24 * np.sqrt(3.0) + abs(float(mr[t])) * 2.0 ** -24
        assert float(mr[t]) + margin >= dist[t] - tol - c, (t, mr[t], dist[t])
        checked += 1
    assert checked > 200


def test_relation_with_segment_nearest(forest):
    """Order-1 trajectories with float32 control points: sqrt(segment d2) lies in [d - tol - eps, d + eps]."""
    pts, half, ix, orc, tr_, t_now, br = forest
    rng = np.random.default_rng(12)
    m = 2000
    a = np.column_stack([rng.uniform(-half, half, m), rng.uniform(-half, half, m), rng.uniform(0.6, 4.0, m)]).astype(np.float32)
    b = (a + rng.normal(size=(m, 3)).astype(np.float32) * 2.0).astype(np.float32)
    tr = dict(traj_first_seg=np.arange(m + 1, dtype=np.int32), seg_order=np.ones(m, np.int32), seg_T=np.ones(m),
              seg_coef_off=np.arange(m + 1, dtype=np.int64) * 6, coef=np.stack([a, b], 2).reshape(m, 6).astype(np.float64).ravel())
    tol = 1e-4
    seg, s, idx, dist = nearest(ix, tr, 0.0, -1.0, tol, 1.0)
    si, sd = ix.segment_nearest(a, b)
    ds = np.sqrt(sd.astype(np.float64))
    eps = ds * 2.0 ** -23 + 1e-9
    assert (seg >= 0).all() and (si >= 0).all()
    assert (ds >= dist - tol - eps).all() and (ds <= dist + eps).all()


def _one(P_list, T_list):
    """CSR arrays of one trajectory from control-point polygons (n+1, 3) and durations."""
    order = np.array([len(P) - 1 for P in P_list], np.int32)
    T = np.array(T_list, np.float64)
    off = np.zeros(len(P_list) + 1, np.int64)
    off[1:] = np.cumsum(3 * (order + 1))
    coef = np.concatenate([(np.asarray(P, np.float64) / T[i]).T.ravel() for i, P in enumerate(P_list)])
    return dict(traj_first_seg=np.array([0, len(P_list)], np.int32), seg_order=order, seg_T=T, seg_coef_off=off, coef=coef)


def _arc(n, center=(0.0, 0.0, 1.0), scale=1.0, seed=0):
    rng = np.random.default_rng(seed)
    base = np.stack([np.linspace(0, 4, n + 1), np.zeros(n + 1), np.zeros(n + 1)], 1)
    base[1:-1, 1] = rng.uniform(0.2, 0.6, n - 1) if n > 1 else 0.0
    return base * scale + np.asarray(center)


def _run_small(pts, tr, t_now, max_range, tol, horizon):
    ix = PointCloudIndex(max_points=max(len(pts), 1), device=0)
    try:
        ix.build(np.asarray(pts, np.float32).reshape(-1, 3))
        out = [nearest(ix, tr, t_now, max_range, tol, horizon, sp) for sp in (L.PC_HOST, L.PC_DEVICE)]
        out.append(nearest(ix, tr, t_now, max_range, tol, horizon))
        for a, b, c in zip(*out):
            assert a.tobytes() == b.tobytes() == c.tobytes()
        return out[0]
    finally:
        ix.close()


def _small_check(pts, tr, t_now, max_range, tol, horizon):
    out = _run_small(pts, tr, t_now, max_range, tol, horizon)
    orc = NB.NearestOracle(pts)
    check_rules(tr, t_now, orc, brackets(orc, tr, t_now, horizon), max_range, tol, horizon, *out)
    return out


def test_curve_through_a_cloud_point():
    tol = 1e-4
    tr = _one([np.array([[0.0, 0.0, 1.0], [4.0, 0.0, 1.0]])], [2.0])
    seg, s, idx, dist = _small_check(np.array([[1.5, 0.0, 1.0], [1.0, 3.0, 1.0]], np.float32), tr, 0.0, -1.0, tol, 10.0)
    assert seg[0] == 0 and idx[0] == 0 and dist[0] <= tol
    for n in (3, 7, 12):
        P = _arc(n, seed=n)
        p = TB.evaluate(P, 0.37).astype(np.float32)
        cast = np.linalg.norm(p.astype(np.float64) - TB.evaluate(P, 0.37))
        seg, s, idx, dist = _small_check(np.array([p, p + 2.0]), _one([P], [2.0]), 0.0, -1.0, tol, 10.0)
        assert idx[0] == 0 and dist[0] <= tol + cast + SLACK


@pytest.mark.parametrize("k", [4, 20])
def test_grazing_points(k):
    r, tol = 0.3, 1e-5
    for n in (1, 3, 7, 12):
        P = _arc(n, seed=n)
        u = np.linspace(0, 1, 200001)
        b = np.array(P)[None].repeat(len(u), 0)
        for _ in range(n):
            b = (1 - u)[:, None, None] * b[:, :-1] + u[:, None, None] * b[:, 1:]
        j = int(np.argmin(np.linalg.norm(b[:, 0] - [2.0, 0.0, 1.0], axis=1)))
        tang = TB.evaluate(P, u[j] + 1e-6) - TB.evaluate(P, u[j] - 1e-6)
        nrm = np.cross(tang, [0.0, 0.0, 1.0])
        nrm /= np.linalg.norm(nrm)
        for dist in (r * (1 - 2.0 ** -k), r * (1 + 2.0 ** -k)):
            p = (b[j, 0] + dist * nrm).astype(np.float32)
            for max_range in (-1.0, r):
                _small_check(p[None], _one([P], [2.0]), 0.0, max_range, tol, 10.0)


def test_minimum_only_in_a_later_segment():
    P1 = _arc(3, seed=1)
    P2 = _arc(5, seed=2) - _arc(5, seed=2)[0] + P1[-1]
    P3 = _arc(4, seed=3) - _arc(4, seed=3)[0] + P2[-1]
    tr = _one([P1, P2, P3], [1.0, 1.5, 0.5])
    late = TB.evaluate(P3, 0.6) + np.array([0.0, 0.0, 0.2])
    far = P1[0] + np.array([0.0, 0.0, 3.0])
    seg, s, idx, dist = _small_check(np.array([far, late], np.float32), tr, 0.0, -1.0, 1e-5, 10.0)
    assert seg[0] == 2 and idx[0] == 1 and abs(dist[0] - 0.2) < 1e-3


def test_t_now_and_horizon_edges():
    Ps = [_arc(2, seed=5), None, None]
    Ps[1] = _arc(4, seed=6) - _arc(4, seed=6)[0] + Ps[0][-1]
    Ps[2] = _arc(6, seed=7) - _arc(6, seed=7)[0] + Ps[1][-1]
    tr = _one(Ps, [0.5, 0.75, 1.0])
    rng = np.random.default_rng(9)
    allp = np.concatenate([TB.evaluate(P, u) for P in Ps for u in np.linspace(0, 1, 9)]).reshape(-1, 3)
    pts = (allp + rng.normal(size=allp.shape) * 0.3).astype(np.float32)
    orc = NB.NearestOracle(pts)
    ix = PointCloudIndex(max_points=len(pts), device=0)
    ix.build(pts)
    try:
        for t_now in (-0.5, 0.5, np.nextafter(0.5, 1.0), 1.25, 2.25, np.nextafter(2.25, 3.0), 5.0, 0.3):
            for horizon in (0.0, -0.25, 0.2, 0.7, 1.25, 3.0):
                for max_range in (-1.0, 0.1):
                    out = [nearest(ix, tr, t_now, max_range, 1e-5, horizon, sp) for sp in (L.PC_HOST, L.PC_DEVICE)]
                    for a, b in zip(*out):
                        assert a.tobytes() == b.tobytes()
                    check_rules(tr, t_now, orc, brackets(orc, tr, t_now, horizon), max_range, 1e-5, horizon, *out[0])
                    if horizon < 0 or t_now > 2.25:
                        assert out[0][0][0] == -1 and out[0][3][0] == np.inf
                    elif max_range < 0:
                        assert out[0][0][0] >= 0
    finally:
        ix.close()


@pytest.mark.parametrize("offset,Tscale", [(1e4, 1.0), (0.0, 1e-3), (0.0, 100.0), (1e4, 100.0)])
def test_offsets_and_time_scales(offset, Tscale):
    tr = synth.bezier_trajectories(60, 8.0, seed=31, order_range=(1, 12))
    tr["seg_T"] = tr["seg_T"] * Tscale
    tr["coef"] = tr["coef"] / Tscale
    for s_ in range(len(tr["seg_order"])):
        n = int(tr["seg_order"][s_])
        o = tr["seg_coef_off"][s_]
        tr["coef"][o:o + 2 * (n + 1)] += offset / tr["seg_T"][s_]
    rng = np.random.default_rng(4)
    pts = np.column_stack([rng.uniform(-8, 8, 60000) + offset, rng.uniform(-8, 8, 60000) + offset, rng.uniform(0.6, 4.0, 60000)])
    pts = pts.astype(np.float32)
    t_now = rng.uniform(-1, 3, 60) * Tscale
    for max_range in (-1.0, 0.2):
        seg, s, idx, dist = _small_check(pts, tr, t_now, max_range, 1e-4, 2.0 * Tscale)
        assert (seg >= 0).sum() > 10


def test_exact_ties_on_a_lattice():
    """Integer lattice, straight and curved trajectories along lattice symmetry lines: many points at exactly the same
    distance; the answer is the same bits in both spaces and on repeat, and satisfies the rules."""
    g = np.arange(-4, 5, dtype=np.float32)
    pts = np.stack(np.meshgrid(g, g, np.arange(0, 4, dtype=np.float32), indexing="ij"), -1).reshape(-1, 3)
    Ps = [np.array([[-3.5, 0.5, 1.5], [3.5, 0.5, 1.5]]), np.array([[-3.0, 0.5, 1.5], [0.0, 0.5, 1.5], [3.0, 0.5, 1.5]]),
          np.array([[0.5, -3.5, 2.5], [0.5, 0.0, 2.5], [0.5, 3.5, 2.5]])]
    for P in Ps:
        for max_range in (-1.0, 0.9):
            seg, s, idx, dist = _small_check(pts, _one([P], [1.0]), 0.0, max_range, 1e-6, 1.0)
            assert seg[0] == 0 and abs(dist[0] - np.sqrt(0.5)) <= 2e-6


def test_empty_index_no_finite_point_and_nan_coefficient():
    tr = synth.bezier_trajectories(20, 8.0, seed=2, order_range=(1, 12))
    for pts in (np.zeros((0, 3), np.float32), np.full((500, 3), np.nan, np.float32),
                np.array([[np.inf, 0, 1], [0, -np.inf, 1], [np.nan, 1, 1]], np.float32)):
        for max_range in (-1.0, 0.5):
            seg, s, idx, dist = _run_small(pts, tr, 0.0, max_range, 1e-3, 5.0)
            assert (seg == -1).all() and (idx == -1).all() and np.isinf(s).all() and np.isinf(dist).all()
    bad = {k: v.copy() for k, v in tr.items()}
    s0 = int(bad["traj_first_seg"][3])
    bad["coef"][bad["seg_coef_off"][s0 + 1] + 1] = np.nan            # trajectory 3's second segment
    pts = np.random.default_rng(0).uniform(-8, 8, (5000, 3)).astype(np.float32)
    seg, s, idx, dist = _run_small(pts, bad, 0.0, -1.0, 1e-3, 100.0)
    assert seg[3] == -1 and idx[3] == -1 and np.isnan(s[3]) and np.isnan(dist[3])
    ok = _run_small(pts, tr, 0.0, -1.0, 1e-3, 100.0)
    for a, b in zip((seg, s, idx, dist), ok):
        assert np.delete(a, 3).tobytes() == np.delete(b, 3).tobytes()


def test_c4_size_batch():
    pts, half = synth.forest_cloud(5_000_000, seed=3, variant="J", return_half=True)
    ix = PointCloudIndex(max_points=len(pts), device=0)
    try:
        ix.build(pts)
        tr = synth.bezier_trajectories(10_000, half * 0.9, seed=8, order_range=(1, 12))
        host = nearest(ix, tr, 0.0, -1.0, 1e-3, 2.0)
        dev = nearest(ix, tr, 0.0, -1.0, 1e-3, 2.0, L.PC_DEVICE)
        for a, b in zip(host, dev):
            assert a.tobytes() == b.tobytes()
        which = np.random.default_rng(1).choice(10_000, 200, replace=False)
        orc = NB.NearestOracle(pts)
        assert check_rules(tr, 0.0, orc, brackets(orc, tr, 0.0, 2.0, which), -1.0, 1e-3, 2.0, *host) == 200
    finally:
        ix.close()


def test_planner_single_trajectory_call(forest):
    pts, half, ix, orc, _, _, _ = forest
    tr = synth.bezier_trajectories(1, half * 0.9, seed=77, order_range=(5, 5), seg_range=(4, 4))
    ix.launches(reset=True)
    out = ix.trajectory_nearest(tr["traj_first_seg"], tr["seg_order"], tr["seg_T"], tr["seg_coef_off"], tr["coef"],
                                1e-3, max_range=1.5, t_now=[0.3], horizon=2.0)
    assert ix.launches() == 1
    check_rules(tr, 0.3, orc, brackets(orc, tr, 0.3, 2.0), 1.5, 1e-3, 2.0, *out)


def nearest_rc(ix, tr, max_range=-1.0, tol=1e-3, horizon=2.0, space=L.PC_HOST, n_traj=None, n_seg=None):
    rec = _traj_records(tr, 0.0)
    n = len(tr["traj_first_seg"]) - 1 if n_traj is None else n_traj
    so, sT = np.ascontiguousarray(tr["seg_order"], np.int32), np.ascontiguousarray(tr["seg_T"], np.float64)
    sc, cf = np.ascontiguousarray(tr["seg_coef_off"], np.int64), np.ascontiguousarray(tr["coef"], np.float64)
    outs = [np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1)), np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1))]
    return ix._L.pc_trajectory_nearest_batch(ix._h, _vp(rec), n, _vp(so), _vp(sT), _vp(sc), len(so) if n_seg is None else n_seg,
                                             _vp(cf), len(cf), space, float(horizon), float(max_range), float(tol),
                                             *[_vp(o) for o in outs])


def _prefix(tr, n):
    """The first n trajectories and only their segments and coefficients."""
    s = int(tr["traj_first_seg"][n])
    off = tr["seg_coef_off"][: s + 1]
    return dict(traj_first_seg=tr["traj_first_seg"][: n + 1], seg_order=tr["seg_order"][:s], seg_T=tr["seg_T"][:s],
                seg_coef_off=off, coef=tr["coef"][: off[-1]])


def staged_bytes(tr, n):
    """What a PC_HOST call on _prefix(tr, n) uploads, each array padded to 256 B: up to 256 KB it travels through one pinned
    staging block, beyond that array by array (pc_traj_upload)."""
    s = int(tr["traj_first_seg"][n])
    pad = lambda b: -(-b // 256) * 256
    return pad(16 * n) + pad(4 * s) + 2 * pad(8 * s) + pad(8 * int(tr["seg_coef_off"][s]))


def test_host_staging_threshold(forest):
    """The last batch that goes through the pinned staging block and the first that does not: PC_HOST returns bit for bit
    what PC_DEVICE returns."""
    pts, half, ix, orc, _, _, _ = forest
    tr = synth.bezier_trajectories(400, half * 0.9, seed=15, order_range=(1, 12))
    size = [staged_bytes(tr, k) for k in range(401)]
    n = max(k for k in range(401) if size[k] <= 1 << 18)
    assert n < 400 and size[n + 1] > 1 << 18
    t_now = _mixed_t_now(400, np.random.default_rng(6))
    for m in (n, n + 1):
        p = _prefix(tr, m)
        host = nearest(ix, p, t_now[:m], 2.0, 1e-3, 2.0)
        dev = nearest(ix, p, t_now[:m], 2.0, 1e-3, 2.0, L.PC_DEVICE)
        for a, b in zip(host, dev):
            assert a.tobytes() == b.tobytes(), f"{m} trajectories"
        assert (host[0] >= 0).any()


def test_refusals(forest):
    pts, half, ix, *_ = forest
    tr = synth.bezier_trajectories(3, 8.0, seed=1)
    assert nearest_rc(ix, tr) == L.PC_OK and nearest_rc(ix, tr, max_range=np.inf) == L.PC_OK
    for kw in (dict(max_range=np.nan), dict(tol=0.0), dict(tol=-1e-3), dict(tol=np.nan), dict(tol=np.inf), dict(horizon=np.nan),
               dict(space=L.PC_HOST_ASYNC), dict(space=L.PC_DEVICE_ASYNC), dict(space=7), dict(n_traj=-1)):
        assert nearest_rc(ix, tr, **kw) == L.PC_EINVAL, kw
    for field, val in (("seg_order", 0), ("seg_order", 13), ("seg_T", 0.0), ("seg_T", np.nan), ("seg_coef_off", -1),
                       ("seg_coef_off", 10 ** 9)):
        bad = {k: v.copy() for k, v in tr.items()}
        bad[field][1] = val
        assert nearest_rc(ix, bad) == L.PC_EINVAL, (field, val)
    bad = {k: v.copy() for k, v in tr.items()}
    bad["traj_first_seg"][-1] += 1
    assert nearest_rc(ix, bad, n_seg=len(tr["seg_order"])) == L.PC_EINVAL
    sh = PointCloudIndex(max_points=len(pts), device=0)
    try:
        sh.build(pts[:1000])
        sh.batch_shard(0, 2)
        assert nearest_rc(sh, tr) == L.PC_EINVAL
    finally:
        sh.close()
