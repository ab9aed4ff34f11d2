"""CPU tests for pc_sphere_sweep_batch: the NULL-handle refusal, and the sweep checker (tests/sweep_brute.c) against a numpy
restatement of the contract's expression, its monotonicity in the radius, and the quadratic branch never rounding to t = 0."""
import numpy as np

from pointcloudtraj_b200 import _lib as L
from sweep_brute import b_clause_rows, brute_sweep, numpy_quadratic_t, numpy_sweep_t, round_down_f32


def test_sweep_null_handle_is_rejected():
    lib = L.load()
    assert lib.pc_sphere_sweep_batch(None, None, None, 0, 3, L.PC_HOST, 0, 0.5, None, None) == L.PC_EINVAL


def _check(pts, a, b, r):
    gi, gt = brute_sweep(pts, a, b, r)
    for j in range(len(a)):
        t = numpy_sweep_t(pts, a[j], b[j], r)
        if not np.isfinite(t).any():
            assert gi[j] == -1 and np.isinf(gt[j]), (j, gi[j], gt[j])
            continue
        o = np.lexsort((np.arange(len(pts)), t))[0]
        assert gi[j] == o and gt[j] == t[o], (j, gi[j], gt[j], o, t[o])


def test_brute_sweep_random_equals_numpy():
    rng = np.random.default_rng(4)
    pts = rng.uniform(-5, 5, (3000, 3)).astype(np.float32)
    a = rng.uniform(-6, 6, (60, 3)).astype(np.float32)
    b = (a + rng.normal(0, 3, (60, 3))).astype(np.float32)
    b[:5] = a[:5]                                       # degenerate segments
    for r in (0.0, 0.05, 0.4, 2.0):
        _check(pts, a, b, r)


def test_brute_sweep_lattice_equals_numpy():
    # spheres swept along and across lattice rows: many points touch at exactly the same t, the lowest index wins
    g = np.arange(8, dtype=np.float32) * 0.5
    pts = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    pts = np.concatenate([pts, pts[::-1]]).astype(np.float32)      # every point twice
    a = np.array([[-1, 0, 0], [-1, 1, 1], [0.25, -1, 0.25], [-1, -1, -1], [3.5, 0, 0], [1, 1, 1]], np.float32)
    b = np.array([[5, 0, 0], [5, 1, 1], [0.25, 5, 0.25], [4, 4, 4], [3.5, 0, 0], [2, 2.5, 0.5]], np.float32)
    for r in (0.0, 0.25, 0.5, 1.0):
        _check(pts, a, b, r)
    gi, gt = brute_sweep(pts, a[:1], b[:1], 0.5)
    assert gi[0] == 0 and gt[0] == 0.5 / 6                # the sphere from x = -1 touches (0, 0, 0) at x = -0.5


def test_brute_sweep_branches_and_nonfinite():
    pts = np.array([[0, 0, 0], [2, 0.3, 0], [4, 0, 0.5], [9, 0, 0]], np.float32)
    a = np.array([[0.1, 0, 0], [1, 0, 0], [5, 0, 0], [np.nan, 0, 0], [0, np.inf, 0], [1, 0, 0]], np.float32)
    b = np.array([[3, 0, 0], [4, 0, 0], [3.6, 0, 0], [1, 0, 0], [0, 0, 0], [1, 0, 0]], np.float32)
    gi, gt = brute_sweep(pts, a, b, 0.5)
    assert gi[0] == 0 and gt[0] == 0.0                      # starts inside
    assert gi[1] == 1 and 0 < gt[1] < 1                     # quadratic branch
    assert np.isnan(gt[3:5]).all() and (gi[3:5] == -1).all()
    assert gi[5] == -1 and np.isinf(gt[5])                  # a == b far from every point
    # the B clause: b exactly 0.5 from a point that the quadratic's rounding may miss, checked against numpy row by row
    _check(pts, a[[0, 1, 2, 5]], b[[0, 1, 2, 5]], 0.5)
    gi, gt = brute_sweep(pts[:0], a[:1], b[:1], 0.5)
    assert gi[0] == -1 and np.isinf(gt[0])
    # contacts that only the B clause reaches: the rounded quadratic lands just above 1
    a, b, p = b_clause_rows(np.random.default_rng(17), 200)
    via_b = 0
    for j in range(200):
        _check(p[j:j + 1], a[j:j + 1], b[j:j + 1], 0.3125)
        via_b += int(numpy_quadratic_t(p[j], a[j], b[j], 0.3125) > 1.0)
    assert via_b > 20


def test_brute_sweep_grazing_equals_numpy():
    # points at lateral distance r (1 + k 2^-26) from 30-50 m segments, far from a: disc changes sign between neighbours
    rng = np.random.default_rng(7)
    a = rng.uniform(-20, 20, (16, 3)).astype(np.float32)
    d = rng.normal(size=(16, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    b = (a + d * rng.uniform(30, 50, (16, 1))).astype(np.float32)
    r = 0.5
    n = np.cross(d, rng.normal(size=(16, 3)))
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    k = np.arange(-8, 9)
    t = rng.uniform(0.3, 0.9, (16, 1))
    p = (a[:, None, :] + t[..., None] * (b - a)[:, None, :] + (r * (1 + k * 2.0 ** -26))[None, :, None] * n[:, None, :])
    pts = p.reshape(-1, 3).astype(np.float32)
    _check(pts, a, b, r)


def test_brute_sweep_monotone_in_radius():
    rng = np.random.default_rng(11)
    pts = rng.uniform(-4, 4, (4000, 3)).astype(np.float32)
    a = rng.uniform(-5, 5, (300, 3)).astype(np.float32)
    b = (a + rng.normal(0, 2.5, (300, 3))).astype(np.float32)
    radii = np.concatenate([[0.0], np.sort(rng.uniform(0, 1.5, 12)), [0.3, np.nextafter(0.3, 1.0)]])
    radii.sort()
    prev = None
    for r in radii:
        gi, gt = brute_sweep(pts, a, b, r)
        f = round_down_f32(gt)
        if prev is not None:
            assert (f <= prev).all(), r                          # t(r1) >= t(r2) for r1 < r2, on the float output
            assert ((prev == np.inf) | (gi >= 0)).all(), r       # contact at r1 implies contact at r2
        prev = f


def test_quadratic_branch_never_rounds_to_zero():
    # points just outside the sphere at a (the smallest h float inputs give) on segments up to 3e38 long (the largest s): every
    # contact through the quadratic branch has t > 0, so t = 0 means c0 <= R2
    rng = np.random.default_rng(3)
    hits = 0
    for r in (2.0 ** -100, 2.0 ** -60, 1e-3, 1.0, 1e3):
        for length in (2.0 ** -90, 1e-3, 1.0, 1e6, 1e30, 3e38):
            a = np.zeros(3, np.float32)
            b = np.array([length, 0, 0], np.float32)
            y = (r * rng.uniform(0, 0.9, 64)).astype(np.float32)                    # lateral offsets inside the radius
            x = np.sqrt(np.maximum(r * r - y.astype(np.float64) ** 2, 0)).astype(np.float32)
            x = np.nextafter(np.nextafter(x, np.float32(np.inf)), np.float32(np.inf))  # just outside the sphere at a
            pts = np.stack([x, y, np.zeros_like(x)], 1)
            t = numpy_sweep_t(pts, a, b, r)
            c0 = pts.astype(np.float64)[:, 0] ** 2 + pts.astype(np.float64)[:, 1] ** 2
            quad = (c0 > r * r) & (t > 0) & (t < 1)
            hits += int(quad.sum())
            assert (t[c0 > r * r] > 0).all(), (r, length)
            gi, gt = brute_sweep(pts, a[None], b[None], r)
            o = np.lexsort((np.arange(len(t)), t))[0]
            assert gt[0] == t[o] and (gi[0] == o or not np.isfinite(t[o]))
    assert hits > 1000, hits


def test_round_down_f32():
    t = np.array([0.0, 1.0, 0.1, 1 / 3, np.inf, np.nan, 2.0 ** -149 * 0.75])
    f = round_down_f32(t)
    ok = np.isfinite(t)
    assert (f[ok].astype(np.float64) <= t[ok]).all()
    assert (np.nextafter(f[ok], np.float32(np.inf)).astype(np.float64) > t[ok]).all()
    assert np.isinf(f[4]) and np.isnan(f[5])
