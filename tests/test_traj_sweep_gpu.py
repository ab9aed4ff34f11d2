"""pc_trajectory_sweep_batch on the GPU: every answer is checked against the numpy oracle of F(rho) (tests/traj_sweep_brute.py)
for the contract's three rules -- nothing earlier than F(r), a witness within r + tol of the reported position (re-evaluated in
fp64 here), and a contact whenever F(r) exists -- with a slack of 1e-9 (distance and time) far below every tol used."""
import ctypes as C

import numpy as np
import pytest

from pointcloudtraj_b200 import PointCloudIndex, PcRadiusParams, synth
from pointcloudtraj_b200 import _lib as L

import traj_sweep_brute as TB

pytestmark = pytest.mark.gpu
SLACK = 1e-9


@pytest.fixture(scope="module")
def forest():
    pts, half = synth.forest_cloud(200_000, seed=11, variant="J", return_half=True)
    ix = PointCloudIndex(max_points=len(pts), device=0)
    ix.build(pts)
    yield pts, half, ix, TB.CloudBoxes(pts)
    ix.close()


def _vp(a):
    return C.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)


def _traj_records(tr, t_now):
    first = tr["traj_first_seg"]
    n = len(first) - 1
    rec = np.zeros(max(n, 1), dtype=np.dtype([("first_seg", "<i4"), ("num_seg", "<i4"), ("t_now", "<f8")]))
    rec["first_seg"][:n], rec["num_seg"][:n], rec["t_now"][:n] = first[:-1], np.diff(first), t_now
    return rec


def sweep(ix, tr, t_now, r, tol, horizon, space=L.PC_HOST):
    """The C call in either space (PC_DEVICE: every array a CUDA tensor), outputs pre-filled with a sentinel."""
    n = len(tr["traj_first_seg"]) - 1
    arrays = [_traj_records(tr, t_now).view(np.uint8), np.ascontiguousarray(tr["seg_order"], np.int32),
              np.ascontiguousarray(tr["seg_T"], np.float64), np.ascontiguousarray(tr["seg_coef_off"], np.int64),
              np.ascontiguousarray(tr["coef"], np.float64)]
    outs = [np.full(n, -7, np.int32), np.full(n, -7.0), np.full(n, -7, np.int32)]
    if space == L.PC_DEVICE:
        import torch
        arrays = [torch.from_numpy(a).cuda() for a in arrays]
        outs = [torch.from_numpy(a).cuda() for a in outs]
        torch.cuda.synchronize()
    rc = ix._L.pc_trajectory_sweep_batch(ix._h, _vp(arrays[0]), n, _vp(arrays[1]), _vp(arrays[2]), _vp(arrays[3]),
                                         len(tr["seg_order"]), _vp(arrays[4]), len(tr["coef"]), space, float(horizon), float(r),
                                         float(tol), *[_vp(o) for o in outs])
    assert rc == L.PC_OK, ix._L.pc_last_error(ix._h)
    if space == L.PC_DEVICE:
        ix.sync()
        outs = [o.cpu().numpy() for o in outs]
    return outs


def check_rules(tr, t_now, cloud, r, tol, horizon, seg, s, idx, which=None):
    """The three rules for trajectories `which` (default: all); returns the number of reported contacts."""
    n = len(tr["traj_first_seg"]) - 1
    t_now = np.broadcast_to(np.asarray(t_now, np.float64), (n,))
    contacts = 0
    for t in (range(n) if which is None else which):
        F = TB.first_contact(tr, t, t_now[t], cloud, r, horizon)
        mot = TB.motion(int(tr["traj_first_seg"][t]), int(tr["traj_first_seg"][t + 1] - tr["traj_first_seg"][t]), float(t_now[t]),
                        tr["seg_T"], horizon)
        if seg[t] < 0:
            assert idx[t] == -1 and s[t] == np.inf, (t, seg[t], s[t], idx[t])
            assert F is None, f"trajectory {t}: contact {F} missed"
            continue
        contacts += 1
        pos = [m[0] for m in mot].index(int(seg[t]))
        sg, sa, sb = mot[pos]
        T = float(tr["seg_T"][sg])
        assert sa <= s[t] <= sb + SLACK * T, (t, s[t], sa, sb)
        if F is not None:
            assert pos < F[0] or (pos == F[0] and s[t] <= F[2] + SLACK * max(T, 1.0)), f"trajectory {t}: {pos, s[t]} after F(r) = {F}"
        P = TB.polygon(tr["coef"], tr["seg_coef_off"], tr["seg_order"], tr["seg_T"], sg)
        k = np.nonzero(cloud.idx == idx[t])[0]
        assert len(k) == 1, f"trajectory {t}: witness {idx[t]} is not a finite cloud point"
        d = np.linalg.norm(TB.evaluate(P, s[t] / T) - cloud.p[k[0]])
        assert d <= r + tol + SLACK, f"trajectory {t}: witness at {d}, r + tol = {r + tol}"
    return contacts


def _mixed_t_now(n, rng):
    t = np.zeros(n)
    sel = rng.random(n) < 0.3
    t[sel] = rng.uniform(-1.0, 4.0, int(sel.sum()))
    return t


@pytest.mark.parametrize("tol", [1e-3, 1e-5])
@pytest.mark.parametrize("r", [0.0, 0.1, 0.5])
def test_forest_rules_both_spaces(forest, r, tol):
    pts, half, ix, cloud = forest
    tr = synth.bezier_trajectories(1000, half * 0.9, seed=21, order_range=(1, 12))
    t_now = _mixed_t_now(1000, np.random.default_rng(5))
    host = sweep(ix, tr, t_now, r, tol, 2.0)
    dev = sweep(ix, tr, t_now, r, tol, 2.0, L.PC_DEVICE)
    again = sweep(ix, tr, t_now, r, tol, 2.0)
    for a, b, c in zip(host, dev, again):
        assert a.tobytes() == b.tobytes() == c.tobytes()
    n = check_rules(tr, t_now, cloud, r, tol, 2.0, *host)
    assert r == 0.0 or n > 100


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


def _run_small(pts, tr, t_now, r, tol, horizon):
    ix = PointCloudIndex(max_points=max(len(pts), 1), device=0)
    try:
        ix.build(np.asarray(pts, np.float32).reshape(-1, 3))
        out = [sweep(ix, tr, t_now, r, tol, horizon, sp) for sp in (L.PC_HOST, L.PC_DEVICE)]
        for a, b in zip(*out):
            assert a.tobytes() == b.tobytes()
        return out[0]
    finally:
        ix.close()


def _closest(P, p):
    u = np.linspace(0, 1, 200001)
    b = np.array(P, np.float64)[None].repeat(len(u), 0)
    for _ in range(len(P) - 1):
        b = (1 - u)[:, None, None] * b[:, :-1] + u[:, None, None] * b[:, 1:]
    d = np.linalg.norm(b[:, 0] - p, axis=1)
    k = int(np.argmin(d))
    return u[k], b[k, 0]


@pytest.mark.parametrize("k", [4, 10, 20])
def test_grazing_points(k):
    r, tol = 0.3, 1e-4
    for n in (1, 3, 7, 12):
        P = _arc(n, seed=n)
        tr = _one([P], [2.0])
        u0, c0 = _closest(P, np.array([2.0, 0.0, 1.0]))
        # a point at distance d from the curve's closest point c0 to (2, 0, 1), along the curve's normal in its plane
        h = 1e-6
        tang = TB.evaluate(P, u0 + h) - TB.evaluate(P, u0 - h)
        nrm = np.cross(tang, [0.0, 0.0, 1.0])
        nrm /= np.linalg.norm(nrm)
        for dist in (r * (1 - 2.0 ** -k), r * (1 + 2.0 ** -k), r + tol / 2):
            p = (c0 + dist * nrm).astype(np.float32)
            seg, s, idx = _run_small(p[None], tr, 0.0, r, tol, 10.0)
            cloud = TB.CloudBoxes(p[None])
            check_rules(tr, 0.0, cloud, r, tol, 10.0, seg, s, idx)
            if dist < r - 1e-6:                                      # beyond the float32 rounding of p: a contact
                assert seg[0] == 0


def test_contact_only_in_a_later_segment_and_start_inside():
    P1 = _arc(3, seed=1)
    P2 = _arc(5, center=P1[-1], seed=2) - _arc(5, seed=2)[0] + 0.0
    P2 = P2 - P2[0] + P1[-1]
    P3 = _arc(4, seed=3) - _arc(4, seed=3)[0] + P2[-1]
    tr = _one([P1, P2, P3], [1.0, 1.5, 0.5])
    late = TB.evaluate(P3, 0.6) + np.array([0.0, 0.0, 0.2])
    pts = np.array([late], np.float32)
    seg, s, idx = _run_small(pts, tr, 0.0, 0.25, 1e-4, 10.0)
    assert seg[0] == 2 and idx[0] == 0
    check_rules(tr, 0.0, TB.CloudBoxes(pts), 0.25, 1e-4, 10.0, seg, s, idx)
    # starting inside contact: the answer is the motion's start
    for t_now in (0.0, 0.4, 1.7):
        mot = TB.motion(0, 3, t_now, tr["seg_T"], 10.0)
        sg, sa, _ = mot[0]
        Pm = [P1, P2, P3][sg]
        c = TB.evaluate(Pm, sa / tr["seg_T"][sg])
        pts = np.array([c + [0.0, 0.1, 0.0], late], np.float32)
        seg, s, idx = _run_small(pts, tr, t_now, 0.25, 1e-4, 10.0)
        assert seg[0] == sg and s[0] == sa and idx[0] == 0


def test_t_now_and_horizon_edges():
    Ps = [_arc(2, seed=5), None, None]
    Ps[1] = _arc(4, seed=6) - _arc(4, seed=6)[0] + Ps[0][-1]
    Ps[2] = _arc(6, seed=7) - _arc(6, seed=7)[0] + Ps[1][-1]
    T = [0.5, 0.75, 1.0]
    tr = _one(Ps, T)
    rng = np.random.default_rng(9)
    allp = np.concatenate([TB.evaluate(P, u) for P in Ps for u in np.linspace(0, 1, 9)]).reshape(-1, 3)
    pts = (allp + rng.normal(size=allp.shape) * 0.3).astype(np.float32)
    cloud = TB.CloudBoxes(pts)
    ix = PointCloudIndex(max_points=len(pts), device=0)
    ix.build(pts)
    try:
        for t_now in (-0.5, 0.5, np.nextafter(0.5, 1.0), 1.25, 2.25, np.nextafter(2.25, 3.0), 5.0, 0.3):
            for horizon in (0.0, -0.25, 0.2, 0.7, 1.25, 3.0):
                for r in (0.05, 0.3):
                    out = [sweep(ix, tr, t_now, r, 1e-4, horizon, sp) for sp in (L.PC_HOST, L.PC_DEVICE)]
                    for a, b in zip(*out):
                        assert a.tobytes() == b.tobytes()
                    check_rules(tr, t_now, cloud, r, 1e-4, horizon, *out[0])
                    if horizon < 0 or t_now > 2.25:
                        assert out[0][0][0] == -1 and out[0][1][0] == np.inf
    finally:
        ix.close()


@pytest.mark.parametrize("offset,Tscale", [(1e4, 1.0), (0.0, 1e-3), (0.0, 100.0), (1e4, 100.0)])
def test_offsets_and_time_scales(offset, Tscale):
    tr = synth.bezier_trajectories(60, 8.0, seed=31, order_range=(1, 12))
    tr["seg_T"] = tr["seg_T"] * Tscale
    tr["coef"] = tr["coef"] / Tscale
    # shift positions by offset: position = T * sum B c, so add offset / T to every coefficient of the x and y blocks
    for s_ in range(len(tr["seg_order"])):
        n = int(tr["seg_order"][s_])
        o = tr["seg_coef_off"][s_]
        tr["coef"][o:o + 2 * (n + 1)] += offset / tr["seg_T"][s_]
    rng = np.random.default_rng(4)
    pts = np.column_stack([rng.uniform(-8, 8, 60000) + offset, rng.uniform(-8, 8, 60000) + offset, rng.uniform(0.6, 4.0, 60000)])
    pts = pts.astype(np.float32)
    t_now = rng.uniform(-1, 3, 60) * Tscale
    r, tol = 0.2, 1e-4
    seg, s, idx = _run_small(pts, tr, t_now, r, tol, 2.0 * Tscale)
    assert check_rules(tr, t_now, TB.CloudBoxes(pts), r, tol, 2.0 * Tscale, seg, s, idx) > 10


def test_empty_index_no_finite_point_and_nan_coefficient():
    tr = synth.bezier_trajectories(20, 8.0, seed=2, order_range=(1, 12))
    for pts in (np.zeros((0, 3), np.float32), np.full((500, 3), np.nan, np.float32),
                np.array([[np.inf, 0, 1], [0, -np.inf, 1], [np.nan, 1, 1]], np.float32)):
        seg, s, idx = _run_small(pts, tr, 0.0, 0.5, 1e-3, 5.0)
        assert (seg == -1).all() and (idx == -1).all() and np.isinf(s).all()
    bad = {k: v.copy() for k, v in tr.items()}
    s0 = int(bad["traj_first_seg"][3])
    bad["coef"][bad["seg_coef_off"][s0 + 1] + 1] = np.nan            # trajectory 3's second segment
    rng = np.random.default_rng(0)
    pts = rng.uniform(-8, 8, (5000, 3)).astype(np.float32)
    seg, s, idx = _run_small(pts, bad, 0.0, 0.01, 1e-3, 100.0)
    assert seg[3] == -1 and idx[3] == -1 and np.isnan(s[3])
    ok, _, _ = _run_small(pts, tr, 0.0, 0.01, 1e-3, 100.0)
    assert (np.delete(seg, 3) == np.delete(ok, 3)).all()


def test_c4_size_batch():
    pts, half = synth.forest_cloud(5_000_000, seed=3, variant="J", return_half=True)
    ix = PointCloudIndex(max_points=len(pts), device=0)
    try:
        ix.build(pts)
        tr = synth.bezier_trajectories(10_000, half * 0.9, seed=8, order_range=(1, 12))
        seg, s, idx = sweep(ix, tr, 0.0, 0.3, 1e-3, 2.0)
        dseg, ds, didx = sweep(ix, tr, 0.0, 0.3, 1e-3, 2.0, L.PC_DEVICE)
        assert seg.tobytes() == dseg.tobytes() and s.tobytes() == ds.tobytes() and idx.tobytes() == didx.tobytes()
        which = np.random.default_rng(1).choice(10_000, 200, replace=False)
        assert check_rules(tr, 0.0, TB.CloudBoxes(pts), 0.3, 1e-3, 2.0, seg, s, idx, which) > 20
    finally:
        ix.close()


def test_planner_single_trajectory_call(forest):
    pts, half, ix, cloud = forest
    tr = synth.bezier_trajectories(1, half * 0.9, seed=77, order_range=(5, 5), seg_range=(4, 4))
    ix.launches(reset=True)
    seg, s, idx = ix.trajectory_sweep(tr["traj_first_seg"], tr["seg_order"], tr["seg_T"], tr["seg_coef_off"], tr["coef"],
                                      0.4, 1e-3, t_now=[0.3], horizon=2.0)
    assert ix.launches() == 1
    check_rules(tr, 0.3, cloud, 0.4, 1e-3, 2.0, seg, s, idx)


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
    pts, half, ix, cloud = forest
    tr = synth.bezier_trajectories(400, half * 0.9, seed=15, order_range=(1, 12))
    size = [staged_bytes(tr, k) for k in range(401)]
    n = max(k for k in range(401) if size[k] <= 1 << 18)
    assert n < 400 and size[n + 1] > 1 << 18
    t_now = _mixed_t_now(400, np.random.default_rng(6))
    for m in (n, n + 1):
        p = _prefix(tr, m)
        host = sweep(ix, p, t_now[:m], 0.3, 1e-3, 2.0)
        dev = sweep(ix, p, t_now[:m], 0.3, 1e-3, 2.0, L.PC_DEVICE)
        for a, b in zip(host, dev):
            assert a.tobytes() == b.tobytes(), f"{m} trajectories"
        assert (host[0] >= 0).any()


def test_refusals(forest):
    pts, half, ix, cloud = forest
    tr = synth.bezier_trajectories(3, 8.0, seed=1)
    ok = lambda **kw: sweep_rc(ix, tr, **kw)
    assert ok() == L.PC_OK
    for kw in (dict(r=-0.1), dict(r=np.nan), dict(r=np.inf), dict(tol=0.0), dict(tol=-1e-3), dict(tol=np.nan), dict(tol=np.inf),
               dict(horizon=np.nan), dict(space=L.PC_HOST_ASYNC), dict(space=L.PC_DEVICE_ASYNC), dict(space=7), dict(n_traj=-1)):
        assert ok(**kw) == L.PC_EINVAL, kw
    for field, val in (("seg_order", 0), ("seg_order", 13), ("seg_T", 0.0), ("seg_T", np.nan), ("seg_coef_off", -1),
                       ("seg_coef_off", 10 ** 9)):
        bad = {k: v.copy() for k, v in tr.items()}
        bad[field][1] = val
        assert sweep_rc(ix, bad) == L.PC_EINVAL, (field, val)
    bad = {k: v.copy() for k, v in tr.items()}
    bad["traj_first_seg"][-1] += 1                                   # the last trajectory runs past the segment arrays
    assert sweep_rc(ix, bad, n_seg=len(tr["seg_order"])) == L.PC_EINVAL
    sh = PointCloudIndex(max_points=len(pts), device=0)
    try:
        sh.build(pts[:1000])
        sh.batch_shard(0, 2)
        assert sweep_rc(sh, tr) == L.PC_EINVAL
    finally:
        sh.close()


def sweep_rc(ix, tr, r=0.3, tol=1e-3, horizon=2.0, space=L.PC_HOST, n_traj=None, n_seg=None):
    rec = _traj_records(tr, 0.0)
    n = len(tr["traj_first_seg"]) - 1 if n_traj is None else n_traj
    so, sT = np.ascontiguousarray(tr["seg_order"], np.int32), np.ascontiguousarray(tr["seg_T"], np.float64)
    sc, cf = np.ascontiguousarray(tr["seg_coef_off"], np.int64), np.ascontiguousarray(tr["coef"], np.float64)
    outs = [np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1)), np.zeros(max(n, 1), np.int32)]
    return ix._L.pc_trajectory_sweep_batch(ix._h, _vp(rec), n, _vp(so), _vp(sT), _vp(sc), len(so) if n_seg is None else n_seg,
                                           _vp(cf), len(cf), space, float(horizon), float(r), float(tol), *[_vp(o) for o in outs])


def test_relation_with_sphere_sweep(forest):
    """Order-1 segments with float32 control points: F(r + tol) <= the answer <= pc_sphere_sweep_batch's contact."""
    pts, half, ix, cloud = forest
    rng = np.random.default_rng(12)
    m = 2000
    a = np.column_stack([rng.uniform(-half, half, m), rng.uniform(-half, half, m), rng.uniform(0.6, 4.0, m)]).astype(np.float32)
    b = (a + rng.normal(size=(m, 3)).astype(np.float32) * 2.0).astype(np.float32)
    T = np.full(m, 1.0)
    tr = dict(traj_first_seg=np.arange(m + 1, dtype=np.int32), seg_order=np.ones(m, np.int32), seg_T=T,
              seg_coef_off=np.arange(m + 1, dtype=np.int64) * 6,
              coef=np.concatenate([np.stack([a, b], 2).reshape(m, 6)], 0).astype(np.float64).ravel())
    r, tol = 0.3, 1e-3
    seg, s, idx = sweep(ix, tr, 0.0, r, tol, 1.0)
    wi, wt = ix.sphere_sweep(a, b, r)
    wi2, wt2 = ix.sphere_sweep(a, b, r + tol)
    hit = wi >= 0
    assert ((seg >= 0) >= hit).all() and ((seg >= 0) <= (wi2 >= 0)).all()
    u = s[seg >= 0]
    assert (u <= np.nextafter(wt[seg >= 0], np.float32(np.inf)).astype(np.float64) + SLACK).all()
    assert (u >= wt2[seg >= 0].astype(np.float64) - SLACK).all()


def test_relation_with_clearance(forest):
    """pc_clearance_batch with search_margin = r - tol: a first hit at a sample is never before the sweep's answer."""
    pts, half, ix, cloud = forest
    tr = synth.bezier_trajectories(300, half * 0.9, seed=41, order_range=(1, 12))
    r, tol, dt, horizon = 0.4, 1e-3, 0.02, 2.0
    seg, s, idx = sweep(ix, tr, 0.0, r, tol, horizon)
    params = PcRadiusParams.make(r - tol, 100.0, -1.0, (0.0, 0.0, 0.0))
    fh, mr, ns = ix.clearance(tr["traj_first_seg"], tr["seg_order"], tr["seg_T"], tr["seg_coef_off"], tr["coef"], params,
                              dt=dt, horizon=horizon)
    first, T = tr["traj_first_seg"], tr["seg_T"]
    for t in range(len(first) - 1):
        if fh[t] < 0:
            continue
        assert seg[t] >= 0, f"trajectory {t}: clearance hit at sample {fh[t]}, no sweep contact"
        # the reference's walk (sim_planning_demo.cpp:735-749) to sample fh[t]
        i, tt, acc, k = 0, 0.0, 0.0, 0
        nseg = int(first[t + 1] - first[t])
        while True:
            Ti = T[first[t] + i]
            if not tt < Ti:
                i, tt = i + 1, 0.0
                continue
            acc += dt
            if acc > horizon:
                i, tt = i + 1, 0.0
                continue
            if k == fh[t]:
                break
            k, tt = k + 1, tt + dt
        sg = int(first[t]) + i
        assert seg[t] < sg or (seg[t] == sg and s[t] <= tt + SLACK), (t, seg[t], s[t], sg, tt)
        assert i < nseg
