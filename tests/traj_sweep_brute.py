"""Independent numpy fp64 oracle of pc_trajectory_sweep_batch's F(rho): the first (segment, local time) of a trajectory's motion
at which a cloud point lies within rho of the sphere's centre.

The motion is the one of the contract (include/pc_index.h): pc_clearance_batch's start (max(0, t_now), then the fp64
segment-skipping loop), then segments in order until the elapsed time -- summed exactly, in rationals -- reaches the horizon.
Per segment the control polygon T * c_j is restricted to the motion by de Casteljau; the points of the hull box dilated by rho
are the candidates; for each, the first root of f(v) = |C(v) - p|^2 - rho^2 is isolated with the Bernstein coefficients of f
(all positive on an interval: no root there), halving intervals earliest first down to 2^-42 of the motion's part of the
segment.  Nothing here shares code with the library."""
from __future__ import annotations

from fractions import Fraction
from math import comb

import numpy as np

LEVELS = 42


def motion(first_seg, num_seg, t_now, seg_T, horizon):
    """[(s, sigma_a, sigma_b), ...] of a trajectory's motion, in time order (empty list: empty motion)."""
    if num_seg <= 0 or not horizon >= 0.0:
        return []
    t_s = t_now if t_now > 0.0 else 0.0
    i = 0
    while i < num_seg:
        if t_s > seg_T[first_seg + i] and i + 1 < num_seg:
            t_s = t_s - seg_T[first_seg + i]
            i += 1
        else:
            break
    if t_s > seg_T[first_seg + i]:
        return []
    out = []
    rem = Fraction(horizon) if np.isfinite(horizon) else None
    for j in range(i, num_seg):
        s = first_seg + j
        T = float(seg_T[s])
        sa = t_s if j == i else 0.0
        if rem is not None and Fraction(sa) + rem < Fraction(T):
            out.append((s, sa, float(Fraction(sa) + rem)))
            break
        out.append((s, sa, T))
        if rem is not None:
            rem -= Fraction(T) - Fraction(sa)
            if rem < 0:
                break
    return out


def polygon(coef, off, order, T, s):
    n = int(order[s])
    c = np.asarray(coef[off[s]:off[s] + 3 * (n + 1)], np.float64).reshape(3, n + 1).T
    return T[s] * c                                   # (n + 1, 3)


def split(P, t):
    """de Casteljau: the control polygons of [0, t] and [t, 1] (last axis any)."""
    n = P.shape[-2] - 1
    left, right = [P[..., 0, :]], [P[..., n, :]]
    b = P
    for _ in range(n):
        b = (1.0 - t) * b[..., :-1, :] + t * b[..., 1:, :]
        left.append(b[..., 0, :])
        right.append(b[..., -1, :])
    return np.stack(left, -2), np.stack(right[::-1], -2)


def restrict(P, ua, ub):
    if ub <= ua:
        _, R = split(P, ua)
        return np.repeat(R[:1], len(P), 0)
    _, R = split(P, ua)
    L, _ = split(R, (ub - ua) / (1.0 - ua)) if ua < 1.0 else (R, None)
    return L


def evaluate(P, u):
    b = np.asarray(P, np.float64)
    for _ in range(len(P) - 1):
        b = (1.0 - u) * b[:-1] + u * b[1:]
    return b[0]


def _first_roots(Q, pts, rho):
    """Earliest v in [0, 1] with |C_Q(v) - p| <= rho, per point (inf: none)."""
    n = len(Q) - 1
    D = Q[None, :, :] - pts[:, None, :]                                   # (m, n+1, 3)
    G = np.einsum("mia,mja->mij", D, D)
    W = np.array([[comb(n, i) * comb(n, j) / comb(2 * n, i + j) for j in range(n + 1)] for i in range(n + 1)])
    f = np.zeros((len(pts), 2 * n + 1))
    for i in range(n + 1):
        for j in range(n + 1):
            f[:, i + j] += W[i, j] * G[:, i, j]
    f -= rho * rho
    best = np.full(len(pts), np.inf)
    cand = np.arange(len(pts))
    lo = np.zeros(len(pts))
    width = 1.0
    for level in range(LEVELS + 1):
        if len(cand) == 0:
            break
        at_lo = f[:, 0] <= 0.0
        np.minimum.at(best, cand[at_lo], lo[at_lo])
        keep = ~at_lo & ~(f > 0.0).all(1) & (lo < best[cand])
        cand, lo, f = cand[keep], lo[keep], f[keep]
        if level == LEVELS:
            np.minimum.at(best, cand, lo)
            break
        fl, fr = split(f[:, :, None], 0.5)
        width *= 0.5
        cand = np.concatenate([cand, cand])
        lo = np.concatenate([lo, lo + width])
        f = np.concatenate([fl[:, :, 0], fr[:, :, 0]])
        order = np.lexsort((lo, cand))
        cand, lo, f = cand[order], lo[order], f[order]
    return best


class CloudBoxes:
    """Cloud points sorted by x for box queries; non-finite points are dropped (they never touch)."""

    def __init__(self, pts):
        p = np.asarray(pts, np.float32)[:, :3].astype(np.float64)
        idx = np.nonzero(np.isfinite(p).all(1))[0]
        o = np.argsort(p[idx, 0], kind="stable")
        self.idx, self.p = idx[o], p[idx[o]]

    def box(self, lo, hi):
        a, b = np.searchsorted(self.p[:, 0], lo[0], side="left"), np.searchsorted(self.p[:, 0], hi[0], side="right")
        sub = self.p[a:b]
        k = (sub[:, 1] >= lo[1]) & (sub[:, 1] <= hi[1]) & (sub[:, 2] >= lo[2]) & (sub[:, 2] <= hi[2])
        return self.idx[a:b][k], sub[k]


def first_contact_segment(P, T, sa, sb, cloud: CloudBoxes, rho):
    """(sigma, point index) of the first contact at radius rho on segment polygon P over local times [sa, sb], or None."""
    ua, ub = sa / T, min(1.0, sb / T)
    Q = restrict(P, ua, ub)
    ids, pts = cloud.box(Q.min(0) - rho, Q.max(0) + rho)
    if len(ids) == 0:
        return None
    v = _first_roots(Q, pts, rho)
    k = int(np.argmin(v))
    if not np.isfinite(v[k]):
        return None
    return T * (ua + v[k] * (ub - ua)), int(ids[k])


def first_contact(tr, t, t_now, cloud: CloudBoxes, rho, horizon):
    """F(rho) of trajectory t of the CSR dict tr (synth.bezier_trajectories layout) as (position of the segment in the motion,
    segment, sigma, point index), or None."""
    first, T = tr["traj_first_seg"], tr["seg_T"]
    mot = motion(int(first[t]), int(first[t + 1] - first[t]), float(t_now), T, horizon)
    for pos, (s, sa, sb) in enumerate(mot):
        r = first_contact_segment(polygon(tr["coef"], tr["seg_coef_off"], tr["seg_order"], T, s), float(T[s]), sa, sb, cloud, rho)
        if r is not None:
            return pos, s, r[0], r[1]
    return None
