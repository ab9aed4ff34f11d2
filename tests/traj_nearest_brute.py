"""Independent numpy fp64 oracle of pc_trajectory_nearest_batch's D*: the infimum over a trajectory's motion of the distance
from the curve to the nearest finite cloud point, returned as a bracket [lo, hi].

The motion and the restricted control polygons are those of tests/traj_sweep_brute.py.  An upper bound comes from sampled
positions (scipy cKDTree); the candidates are the points in each restricted polygon's hull box dilated by it; per candidate,
min_v |C(v) - p|^2 is bracketed with the Bernstein coefficients of |C(v) - p|^2 (the end coefficients are values of the
curve, the smallest coefficient bounds the interval from below), halving the intervals that can still hold the minimum down
to 2^-42 of the motion's part of a segment, or until the bracket is as tight as fp64 allows.  Nothing here shares code with
the library."""
from __future__ import annotations

from math import comb

import numpy as np
from scipy.spatial import cKDTree

import traj_sweep_brute as TB

LEVELS = 42
SAMPLES = 65
EPS = np.finfo(np.float64).eps


def _bernstein_sq(Q, pts):
    """Bernstein coefficients (degree 2n) of |C_Q(v) - p|^2 for each p, and the magnitude that bounds their rounding."""
    n = len(Q) - 1
    D = Q[None, :, :] - pts[:, None, :]
    G = np.einsum("mia,mja->mij", D, D)
    W = np.array([[comb(n, i) * comb(n, j) / comb(2 * n, i + j) for j in range(n + 1)] for i in range(n + 1)])
    f = np.zeros((len(pts), 2 * n + 1))
    for i in range(n + 1):
        for j in range(n + 1):
            f[:, i + j] += W[i, j] * G[:, i, j]
    return f, float(np.abs(G).max()) if len(pts) else 0.0


def _halves(f):
    """de Casteljau at 1/2 of the rows of f: the coefficients of both halves."""
    left, right = [f[:, 0]], [f[:, -1]]
    b = f
    for _ in range(f.shape[1] - 1):
        b = 0.5 * (b[:, :-1] + b[:, 1:])
        left.append(b[:, 0])
        right.append(b[:, -1])
    return np.stack(left, 1), np.stack(right[::-1], 1)


def _parts(tr, t, t_now, horizon):
    first, T = tr["traj_first_seg"], tr["seg_T"]
    mot = TB.motion(int(first[t]), int(first[t + 1] - first[t]), float(t_now), T, horizon)
    out = []
    for s, sa, sb in mot:
        P = TB.polygon(tr["coef"], tr["seg_coef_off"], tr["seg_order"], T, s)
        Ts = float(T[s])
        out.append(TB.restrict(P, sa / Ts, min(1.0, sb / Ts)))
    return out


class NearestOracle:
    def __init__(self, pts):
        self.cloud = TB.CloudBoxes(pts)
        self.tree = cKDTree(self.cloud.p) if len(self.cloud.p) else None

    def bracket(self, tr, t, t_now, horizon):
        """(lo, hi) with lo <= D* <= hi for trajectory t of the CSR dict tr; (inf, inf) for an empty motion or cloud."""
        parts = _parts(tr, t, t_now, horizon)
        if not parts or self.tree is None:
            return np.inf, np.inf
        u = np.linspace(0.0, 1.0, SAMPLES)
        hi = np.inf
        for Q in parts:
            X = np.stack([TB.evaluate(Q, v) for v in u])
            hi = min(hi, float(self.tree.query(X)[0].min()))
        state, err = [], 0.0
        for Q in parts:
            ids, pts = self.cloud.box(Q.min(0) - hi, Q.max(0) + hi)
            if len(ids):
                f, g = _bernstein_sq(Q, pts)
                err = max(err, 64 * EPS * g * (2 * len(Q)))
                state.append(f)
        hi2 = hi * hi
        lo2 = hi2
        for level in range(LEVELS + 1):
            lb = np.inf
            for f in state:
                if len(f):
                    hi2 = min(hi2, float(f[:, 0].min()), float(f[:, -1].min()))
                    lb = min(lb, float(f.min()))
            lo2 = min(lb, hi2)
            if level == LEVELS or hi2 - lo2 <= 2 * err or np.sqrt(hi2) - np.sqrt(max(lo2, 0.0)) <= 1e-11:
                break
            nxt = []
            for f in state:
                keep = f.min(1) - err <= hi2 + err
                fl, fr = _halves(f[keep])
                nxt.append(np.concatenate([fl, fr]))
            state = nxt
        return float(np.sqrt(max(lo2 - err, 0.0))), float(np.sqrt(hi2 + err))
