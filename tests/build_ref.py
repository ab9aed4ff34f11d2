"""Plain numpy restatement of pc_index_build (pointcloudtraj_b200/csrc/build_kernels.cuh, common.cuh, pc_index.cu), written
from the rules of the build rather than from its GPU code paths, to check the built index record for record.

All arithmetic is float32 with one rounding per operation, as the kernels do it:
  * bits per axis: 10 up to 4 Mi points, then one more for every 4x more points (pc_key_bits_per_axis);
  * frame: lo / hi = per-axis min / max over the points whose three coordinates are all finite, ext = max(hi - lo),
    inv = float32(2^bits) * (1 - 1e-6f) / ext when 0 < ext < inf, else 0;
  * cell: fmin(fmax((v - lo) * inv, 0), 2^bits - 1) truncated (NaN -> 0, as fmaxf does);
  * key: Skilling's Hilbert transform with `bits` bits per axis, interleaved axis 0 highest (pc_hilbert30_cells, pc_hilbert63);
  * curve order: stable sort of the keys; points = (x, y, z, index bits) in curve order plus PC_LEAF copies of the last point;
  * tree: built top-down, node [f, l] split at the highest bit where (key, position) of f and l differ, children s and s + 1,
    a child of <= PC_LEAF points is the leaf PC_REF_LEAF | first, boxes = fmin / fmax over the child's points (NaN ignored);
  * seeds: the breadth-first frontier of pc_tree_seed_kernel.
"""
from __future__ import annotations

import numpy as np

PC_LEAF = 4
PC_REF_LEAF = 0x80000000
SEED_WORDS, SEED_INNER, SEED_LEAF = 100, 2, 34


def key_bits_per_axis(n: int) -> int:
    b, lim = 10, 1 << 22
    while n > lim and b < 21:
        b += 1
        lim <<= 2
    return b


def frame(xyz: np.ndarray):
    """-> (lo[3], hi[3], inv) as float32.  A cloud without a finite point has lo = +inf, hi = -inf and inv = 0."""
    p = np.asarray(xyz, np.float32)[:, :3]
    fin = np.isfinite(p).all(1)
    lo = np.full(3, np.inf, np.float32)
    hi = np.full(3, -np.inf, np.float32)
    if fin.any():
        lo, hi = p[fin].min(0), p[fin].max(0)
    return lo, hi, _inv_cell(lo, hi, key_bits_per_axis(len(p)))


def _inv_cell(lo, hi, bits):
    with np.errstate(invalid="ignore", over="ignore"):
        ext = np.float32(0)
        for a in range(3):
            ext = np.fmax(ext, np.float32(hi[a] - lo[a]))
    if not (ext > 0 and ext < np.inf):
        return np.float32(0)
    return np.float32(np.float32(np.float32(1 << bits) * np.float32(np.float32(1) - np.float32(1e-6))) / ext)


def cells(xyz: np.ndarray, lo, inv, bits) -> np.ndarray:
    """(n, 3) uint32 cell coordinates in the frame (lo, inv)."""
    p = np.asarray(xyz, np.float32)[:, :3]
    with np.errstate(invalid="ignore", over="ignore"):
        c = (p - lo.astype(np.float32)) * np.float32(inv)
    c = np.fmin(np.fmax(c, np.float32(0)), np.float32((1 << bits) - 1))
    return c.astype(np.uint32)


def hilbert_keys(c: np.ndarray, bits: int) -> np.ndarray:
    """Skilling's transform of (n, 3) cells with `bits` bits per axis -> uint64 keys of 3 * bits bits."""
    X = [c[:, a].astype(np.uint32) for a in range(3)]
    Q = 1 << (bits - 1)
    while Q > 1:
        P = np.uint32(Q - 1)
        for i in range(3):
            m = (X[i] & np.uint32(Q)) != 0
            t = np.where(m, np.uint32(0), (X[0] ^ X[i]) & P)
            X[0] = np.where(m, X[0] ^ P, X[0] ^ t)
            if i:
                X[i] = X[i] ^ t
        Q >>= 1
    X[1] = X[1] ^ X[0]
    X[2] = X[2] ^ X[1]
    t = np.zeros_like(X[2])
    Q = 1 << (bits - 1)
    while Q > 1:
        t ^= np.where((X[2] & np.uint32(Q)) != 0, np.uint32(Q - 1), np.uint32(0))
        Q >>= 1
    key = np.zeros(len(c), np.uint64)
    for j in range(bits):
        for a in range(3):
            bit = ((X[a] ^ t) >> np.uint32(j)) & np.uint32(1)
            key |= bit.astype(np.uint64) << np.uint64(3 * j + 2 - a)
    return key


def _highest_bit(v: np.ndarray) -> np.ndarray:
    """index of the highest set bit of nonzero uint64 values"""
    v = v.astype(np.uint64)
    r = np.zeros(len(v), np.int64)
    for s in (32, 16, 8, 4, 2, 1):
        big = (v >> np.uint64(s)) != 0
        r += np.where(big, s, 0)
        v = np.where(big, v >> np.uint64(s), v)
    return r


class BuildRef:
    """The index pc_index_build makes of `xyz` ((n, 3) or (n, 4) float32; only x, y, z are read).

    Attributes: n, bits, lo, hi, inv, keys (sorted, uint64), order (curve position -> input index), points (uint32 (n + 4, 4)),
    n_nodes, root, root_count, records (uint32 (n_nodes, 16), zero where unreachable), reachable (bool (n_nodes,)),
    first / last / split / depth (int64 (n_nodes,), -1 where unreachable), seeds (uint32 (100,)), seed_mask (bool (100,)).
    """

    def __init__(self, xyz: np.ndarray):
        p = np.ascontiguousarray(np.asarray(xyz, np.float32)[:, :3])
        n = self.n = len(p)
        self.bits = key_bits_per_axis(n)
        self.lo, self.hi, self.inv = frame(p)
        keys = hilbert_keys(cells(p, self.lo, self.inv, self.bits), self.bits)
        self.order = np.argsort(keys, kind="stable")
        self.keys = keys[self.order]
        sp = p[self.order]
        pts = np.empty((n + PC_LEAF, 4), np.uint32)
        pts[:n, :3] = sp.view(np.uint32)
        pts[:n, 3] = self.order.astype(np.uint32)
        pts[n:] = pts[n - 1]
        self.points = pts
        self.n_nodes = n - 1 if n > PC_LEAF else 0
        self.root = 0 if self.n_nodes else PC_REF_LEAF
        self.root_count = 0 if self.n_nodes else n
        self._tree(sp)
        self._seeds()

    # ---- tree ------------------------------------------------------------------------------------------------------------
    def _split(self, f, l):
        kf, kl = self.keys[f], self.keys[l]
        s = np.empty(len(f), np.int64)
        d = kf != kl
        if d.any():
            b = _highest_bit(kf[d] ^ kl[d]).astype(np.uint64)
            bound = ((kf[d] >> b) + np.uint64(1)) << b          # first key above f's prefix
            s[d] = np.searchsorted(self.keys, bound, side="left") - 1
        e = ~d
        if e.any():
            b = _highest_bit((f[e] ^ l[e]).astype(np.uint64))
            s[e] = ((l[e] >> b) << b) - 1
        return s

    def _tree(self, sp):
        m = self.n_nodes
        self.records = np.zeros((m, 16), np.uint32)
        self.reachable = np.zeros(m, bool)
        self.first, self.last, self.split, self.depth = (np.full(m, -1, np.int64) for _ in range(4))
        if m == 0:
            return
        levels = []
        ids, f, l = np.zeros(1, np.int64), np.zeros(1, np.int64), np.full(1, self.n - 1, np.int64)
        depth = 0
        while len(ids):
            s = self._split(f, l)
            assert ((s >= f) & (s < l)).all()
            self.reachable[ids] = True
            self.first[ids], self.last[ids], self.split[ids], self.depth[ids] = f, l, s, depth
            cf = (f, s + 1)
            cl = (s, l)
            for c in range(2):
                cnt = cl[c] - cf[c] + 1
                leaf = cnt <= PC_LEAF
                ref = np.where(leaf, PC_REF_LEAF | cf[c], s + c).astype(np.uint32)
                self.records[ids, 6 + c] = ref
                self.records[ids, 14 + c] = cnt.astype(np.uint32)
            levels.append(ids)
            nf, nl, ni = [], [], []
            for c in range(2):
                inner = cl[c] - cf[c] + 1 > PC_LEAF
                nf.append(cf[c][inner]); nl.append(cl[c][inner]); ni.append((s + c)[inner])
            ids, f, l = np.concatenate(ni), np.concatenate(nf), np.concatenate(nl)
            depth += 1
        # boxes: leaves partition [0, n), so one reduceat over the leaf starts gives every leaf box; inner boxes bottom-up
        refs = self.records[self.reachable][:, 6:8].ravel()
        starts = np.sort((refs[(refs & PC_REF_LEAF) != 0] & 0x7fffffff).astype(np.int64))
        assert starts[0] == 0 and len(np.unique(starts)) == len(starts)
        lo_in = np.where(np.isnan(sp), np.float32(np.inf), sp)
        hi_in = np.where(np.isnan(sp), np.float32(-np.inf), sp)
        leaf_lo = np.minimum.reduceat(lo_in, starts, axis=0)
        leaf_hi = np.maximum.reduceat(hi_in, starts, axis=0)
        node_lo = np.zeros((m, 3), np.float32)
        node_hi = np.zeros((m, 3), np.float32)
        rec_f = self.records.view(np.float32)
        for ids in reversed(levels):
            bl, bh = [], []
            for c in range(2):
                ref = self.records[ids, 6 + c]
                leaf = (ref & PC_REF_LEAF) != 0
                src = np.where(leaf, 0, ref).astype(np.int64)
                clo, chi = node_lo[src], node_hi[src]
                k = np.searchsorted(starts, (ref[leaf] & 0x7fffffff).astype(np.int64))
                clo[leaf], chi[leaf] = leaf_lo[k], leaf_hi[k]
                for a in range(3):
                    rec_f[ids, 2 * a + c] = clo[:, a]
                    rec_f[ids, 8 + 2 * a + c] = chi[:, a]
                bl.append(clo); bh.append(chi)
            node_lo[ids] = np.minimum(bl[0], bl[1])
            node_hi[ids] = np.maximum(bh[0], bh[1])

    # ---- seeds -----------------------------------------------------------------------------------------------------------
    def _seeds(self):
        seeds = np.zeros(SEED_WORDS, np.uint32)
        cur, leaf = [], []
        if self.root & PC_REF_LEAF:
            leaf.append((self.root, self.root_count))
        else:
            cur.append(self.root)
        while cur and 2 * len(cur) <= 32 and len(leaf) + 2 * len(cur) <= 32:
            nxt = []
            for c in range(2):
                for node in cur:
                    r, k = int(self.records[node, 6 + c]), int(self.records[node, 14 + c])
                    if r & PC_REF_LEAF:
                        leaf.append((r, k))
                    else:
                        nxt.append(r)
            cur = nxt
        seeds[0], seeds[1] = len(cur), len(leaf)
        seeds[SEED_INNER:SEED_INNER + len(cur)] = cur
        for j, (r, k) in enumerate(leaf):
            seeds[SEED_LEAF + 2 * j], seeds[SEED_LEAF + 2 * j + 1] = r, k
        mask = np.zeros(SEED_WORDS, bool)
        mask[:2] = True
        mask[SEED_INNER:SEED_INNER + len(cur)] = True
        mask[SEED_LEAF:SEED_LEAF + 2 * len(leaf)] = True
        self.seeds, self.seed_mask = seeds, mask
