"""Host-side mirror of the kd-tree interface over the GPU index (thin wrapper over the C ABI).

Names follow the reference: ``build`` = kd_clear + n x kd_insert3 (Utils/kdtree/src/kdtree.c:143-159,
244-251), ``nearest`` = kd_nearest3 (:493-500), ``range`` = kd_nearest_range3 (:595-602), ``radius`` =
safeRegionRrtStar::radiusSearch (Planner/src/corridor_finder.cpp:113-133), ``clearance`` =
checkSafeTrajectory (Planner/src/sim_planning_demo.cpp:729-781).

Inputs are numpy arrays (PC_HOST: results come back as numpy arrays, the call returns when they are
resident) or torch CUDA tensors (PC_DEVICE: results are torch tensors; the call is asynchronous when the
handle was created on torch's stream, and blocking when it has a private stream).  All computation happens in libpcindex.so; nothing here computes distances.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


def _is_torch(a):
    return type(a).__module__.startswith("torch")


class PointCloudIndex:
    def __init__(self, max_points: int = 0, device: int = 0, stream=None):
        """stream: raw cudaStream_t (int) or None for a private stream; pass
        ``torch.cuda.current_stream().cuda_stream`` to order the calls with torch work."""
        self._L = L.load()
        h = C.c_void_p()
        # torch tensors are produced and consumed on torch's current stream; a handle with a PRIVATE stream (stream=None) is
        # not ordered with it, so torch-mode calls on such a handle synchronise on both sides (see _torch_fence)
        self._private_stream = stream is None
        if stream is not None and int(stream) == 0:
            stream = 1      # cudaStreamLegacy: NULL means "create a private stream" in the C ABI
        rc = self._L.pc_index_create(C.byref(h), int(device), int(max_points), C.c_void_p(stream or 0))
        if rc != L.PC_OK:
            raise L.PcError(rc, self._L.pc_last_error(None).decode())
        self._h = h
        self.device = int(device)

    # ---- plumbing ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._L.pc_index_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, ok=(L.PC_OK,)):
        if rc not in ok:
            raise L.PcError(rc, self._L.pc_last_error(self._h).decode())
        return rc

    def _rows(self, a, name):
        """-> (pointer, n, stride, space, keepalive, torch_mode)"""
        if _is_torch(a):
            import torch
            if not a.is_cuda:
                raise TypeError(f"{name}: torch tensors must live on the GPU (use numpy for host data)")
            if a.dtype != torch.float32 or a.dim() != 2 or a.shape[1] not in (3, 4):
                raise TypeError(f"{name}: expected float32 (n, 3|4)")
            a = a.contiguous()
            return C.c_void_p(a.data_ptr()), a.shape[0], a.shape[1], L.PC_DEVICE, a, True
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.ndim != 2 or a.shape[1] not in (3, 4):
            raise TypeError(f"{name}: expected float32 (n, 3|4)")
        return C.c_void_p(a.ctypes.data), a.shape[0], a.shape[1], L.PC_HOST, a, False

    def _torch_fence(self, torch_mode, after=False):
        """Handle created without a stream + torch tensors: wait for torch's stream before the call (inputs, output pre-fills)
        and for the handle's stream after it (results), so that correctness never depends on the caller passing a stream."""
        if torch_mode and self._private_stream:
            if after:
                self.sync()
            else:
                import torch
                torch.cuda.current_stream(self.device).synchronize()

    NOT_MINE_IDX = -2 ** 31        # shard mode: pre-fill of entries owned by other ranks (float outputs: NaN)

    def _out(self, m, dtype, torch_mode, ref=None):
        shard = getattr(self, "_shard_n", 1) > 1
        fill = (self.NOT_MINE_IDX if dtype == np.int32 else float("nan")) if shard else None
        if torch_mode:
            import torch
            tdt = {np.int32: torch.int32, np.float32: torch.float32, np.int64: torch.int64}[dtype]
            t = torch.empty(m, dtype=tdt, device=ref.device) if fill is None else torch.full((m,), fill, dtype=tdt, device=ref.device)
            return t, C.c_void_p(t.data_ptr())
        a = np.empty(m, dtype=dtype) if fill is None else np.full(m, fill, dtype=dtype)
        return a, C.c_void_p(a.ctypes.data)

    # ---- index ------------------------------------------------------------------------------------
    def build(self, xyz):
        """Rebuild the index from scratch (kd_clear + n x kd_insert3); point i keeps identity i."""
        p, n, stride, space, keep, tm = self._rows(xyz, "xyz")
        self._torch_fence(tm)
        self._check(self._L.pc_index_build(self._h, p, n, stride, space))
        self._torch_fence(tm, after=True)
        self._cloud_keepalive = keep
        return self

    @property
    def size(self):
        return int(self._L.pc_index_size(self._h))

    def sync(self):
        self._check(self._L.pc_index_sync(self._h))

    def last_build_ms(self):
        ms = C.c_float(0)
        self._check(self._L.pc_index_last_build_ms(self._h, C.byref(ms)))
        return ms.value

    def view(self):
        v = L.PcIndexView()
        self._check(self._L.pc_index_view_get(self._h, C.byref(v)))
        return v

    def launches(self, reset=False):
        return int(self._L.pc_launch_count(self._h, 1 if reset else 0))

    def batch_shard(self, rank=0, n_ranks=1):
        """Spatial sharding (pc_batch_shard): every rank passes the same batch, each answers its stretch of the curve."""
        self._check(self._L.pc_batch_shard(self._h, int(rank), int(n_ranks)))
        self._shard_n = int(n_ranks)

    def set_radius_arith(self, mode):
        """PC_ARITH_FP64 (default) or PC_ARITH_PCL_FLOAT: arithmetic of the radiusSearch epilogue (pc_index.h)."""
        self._check(self._L.pc_index_set_radius_arith(self._h, int(mode)))

    def profile(self, on=True):
        self._check(self._L.pc_profile_enable(self._h, 1 if on else 0))

    def last_batch_ms(self):
        """(ordering ms, search-kernel ms) of the last PC_DEVICE batch (needs profile(True))."""
        a, b = C.c_float(0), C.c_float(0)
        self._check(self._L.pc_profile_last_batch(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    # ---- queries ----------------------------------------------------------------------------------
    def nearest(self, q, flags=L.PC_QUERY_AUTO, want_idx=True, want_d2=True):
        """kd_nearest3 for every row of q.  Returns (idx int32, d2 float32); idx -1 / d2 inf when empty."""
        p, m, stride, space, keep, tm = self._rows(q, "q")
        idx, pi = self._out(m, np.int32, tm, keep) if want_idx else (None, C.c_void_p(0))
        d2, pd = self._out(m, np.float32, tm, keep) if want_d2 else (None, C.c_void_p(0))
        self._torch_fence(tm)
        self._check(self._L.pc_nearest_batch(self._h, p, m, stride, space, flags, pi, pd))
        self._torch_fence(tm, after=True)
        return idx, d2

    def knn(self, q, k, max_range=None, flags=L.PC_QUERY_AUTO):
        """The k nearest points of every row of q (pcl nearestKSearch; with max_range, radiusSearch(q, max_range, ..., k)).
        Returns (idx int32 (m, k), d2 float32 (m, k)), each row ascending by (d2, index), padded with -1 / inf."""
        p, m, stride, space, keep, tm = self._rows(q, "q")
        k = int(k)
        idx, pi = self._out(m * k, np.int32, tm, keep)
        d2, pd = self._out(m * k, np.float32, tm, keep)
        r = -1.0 if max_range is None else float(max_range)
        self._torch_fence(tm)
        self._check(self._L.pc_knn_batch(self._h, p, m, stride, space, int(flags), k, r, pi, pd))
        self._torch_fence(tm, after=True)
        return idx.reshape(m, k), d2.reshape(m, k)

    def knn_large(self, q, k, max_range=None, flags=L.PC_QUERY_AUTO):
        """knn() for k up to PC_KNN_LARGE_MAX (pc_knn_large_batch; pcl nearestKSearch with any k a kd-tree user asks for).
        Returns (idx int32 (m, k), d2 float32 (m, k)), each row ascending by (d2, index), padded with -1 / inf; numpy queries give
        numpy arrays, torch CUDA tensors give tensors."""
        p, m, stride, space, keep, tm = self._rows(q, "q")
        k = int(k)
        idx, pi = self._out(m * k, np.int32, tm, keep)
        d2, pd = self._out(m * k, np.float32, tm, keep)
        r = -1.0 if max_range is None else float(max_range)
        self._torch_fence(tm)
        self._check(self._L.pc_knn_large_batch(self._h, p, m, stride, space, int(flags), k, r, pi, pd))
        self._torch_fence(tm, after=True)
        return idx.reshape(m, k), d2.reshape(m, k)

    def segment_nearest(self, a, b, max_range=None, flags=L.PC_QUERY_AUTO):
        """The nearest cloud point to every segment [a[i], b[i]] (pc_segment_nearest_batch); with max_range only points within
        it.  Returns (idx int32, d2 float32): -1 / inf where no point counts, -1 / NaN for a non-finite endpoint.  a and b are
        both numpy arrays or both torch CUDA tensors of the same shape."""
        pa, m, stride, space, keep_a, tm = self._rows(a, "a")
        pb, mb, stride_b, space_b, keep_b, _ = self._rows(b, "b")
        if (mb, stride_b, space_b) != (m, stride, space):
            raise ValueError("segment_nearest: a and b need the same shape and memory space")
        idx, pi = self._out(m, np.int32, tm, keep_a)
        d2, pd = self._out(m, np.float32, tm, keep_a)
        r = -1.0 if max_range is None else float(max_range)
        self._torch_fence(tm)
        self._check(self._L.pc_segment_nearest_batch(self._h, pa, pb, m, stride, space, int(flags), r, pi, pd))
        self._torch_fence(tm, after=True)
        return idx, d2

    def radius(self, q, params: L.PcRadiusParams, flags=L.PC_RADIUS_BOUNDED, want_idx=False):
        """safeRegionRrtStar::radiusSearch for every row of q.  Returns radius float32 (and idx int32)."""
        p, m, stride, space, keep, tm = self._rows(q, "q")
        r, pr = self._out(m, np.float32, tm, keep)
        idx, pi = self._out(m, np.int32, tm, keep) if want_idx else (None, C.c_void_p(0))
        self._torch_fence(tm)
        self._check(self._L.pc_radius_batch(self._h, p, m, stride, space, flags, C.byref(params), pr, pi))
        self._torch_fence(tm, after=True)
        return (r, idx) if want_idx else r

    def radius_async(self, q_pinned, out_pinned, params: L.PcRadiusParams, flags=L.PC_RADIUS_BOUNDED):
        """PC_HOST_ASYNC radius batch: q_pinned / out_pinned are numpy views of PINNED host memory (float32 (m,3|4) and
        float32 (m,)); the call only enqueues the batch, results are valid after sync().  Give every batch in flight
        its own buffers."""
        if q_pinned.dtype != np.float32 or q_pinned.ndim != 2 or not q_pinned.flags.c_contiguous:
            raise TypeError("q_pinned: contiguous float32 (m, 3|4)")
        m, stride = q_pinned.shape
        self._check(self._L.pc_radius_batch(self._h, C.c_void_p(q_pinned.ctypes.data), m, stride, L.PC_HOST_ASYNC, flags,
                                            C.byref(params), C.c_void_p(out_pinned.ctypes.data), C.c_void_p(0)))

    def check_traj_pt_col(self, pts, params: L.PcRadiusParams):
        """safeRegionRrtStar::checkTrajPtCol (corridor_finder.cpp:412-416): radiusSearch(pt) < 0."""
        return self.radius(pts, params) < 0

    def range(self, q, r, cap=None):
        """kd_nearest_range3 for every row of q (host arrays).  Returns (offsets int64[m+1], idx int32[total]),
        each list ascending by original index."""
        p, m, stride, space, keep, tm = self._rows(q, "q")
        if tm:
            raise TypeError("range(): host (numpy) queries only")
        rr = np.ascontiguousarray(np.atleast_1d(r), dtype=np.float64)
        scalar = 1 if rr.shape[0] == 1 else 0
        if not scalar and rr.shape[0] != m:
            raise ValueError("range: need one radius or one per query")
        off = np.zeros(m + 1, dtype=np.int64)
        pr = C.c_void_p(rr.ctypes.data)
        if cap is None:
            self._check(self._L.pc_range_batch(self._h, p, m, stride, space, pr, scalar, C.c_void_p(off.ctypes.data), C.c_void_p(0), 0))
            cap = int(off[-1])
        out = np.empty(max(cap, 1), dtype=np.int32)
        rc = self._L.pc_range_batch(self._h, p, m, stride, space, pr, scalar, C.c_void_p(off.ctypes.data), C.c_void_p(out.ctypes.data), cap)
        self._check(rc, ok=(L.PC_OK, L.PC_ECAP))
        if rc == L.PC_ECAP:
            raise L.PcError(rc, f"range: {int(off[-1])} hits exceed cap {cap}")
        return off, out[: int(off[-1])]

    def range_sorted(self, q, r, max_nn=0, cap=None):
        """pcl radiusSearch(q, r, k_indices, k_sqr_distances, max_nn) for every row of q (pc_range_sorted_batch).  r: one
        radius or one per query; max_nn = 0 keeps every hit.  Returns (offsets int64[m+1], idx int32[total], d2 float32[total]),
        each row ascending by (d2, index) and cut to max_nn.  numpy queries give numpy arrays; torch CUDA tensors give tensors
        (sized by an offsets-only call first)."""
        p, m, stride, space, keep, tm = self._rows(q, "q")
        max_nn = int(max_nn)
        if tm:
            import torch
            rr = torch.as_tensor(r, dtype=torch.float64, device=keep.device).reshape(-1).contiguous()
            n_r, pr = rr.shape[0], C.c_void_p(rr.data_ptr())
            off = torch.zeros(m + 1, dtype=torch.int64, device=keep.device)
            poff = C.c_void_p(off.data_ptr())
        else:
            rr = np.ascontiguousarray(np.atleast_1d(r), dtype=np.float64)
            n_r, pr = rr.shape[0], C.c_void_p(rr.ctypes.data)
            off = np.zeros(m + 1, dtype=np.int64)
            poff = C.c_void_p(off.ctypes.data)
        scalar = 1 if n_r == 1 else 0
        if not scalar and n_r != m:
            raise ValueError("range_sorted: need one radius or one per query")
        call = lambda pi, pd, c: self._L.pc_range_sorted_batch(self._h, p, m, stride, space, pr, scalar, max_nn, poff, pi, pd, c)
        self._torch_fence(tm)
        if cap is None:
            self._check(call(C.c_void_p(0), C.c_void_p(0), 0))
            self._torch_fence(tm, after=True)
            cap = int(off[-1])
        cap = int(cap)
        idx, pi = self._out(max(cap, 1), np.int32, tm, keep)
        d2, pd = self._out(max(cap, 1), np.float32, tm, keep)
        rc = call(pi, pd, cap)
        self._torch_fence(tm, after=True)
        self._check(rc, ok=(L.PC_OK, L.PC_ECAP))
        total = int(off[-1])
        if rc == L.PC_ECAP:
            raise L.PcError(rc, f"range_sorted: {total} hits exceed cap {cap}")
        return off, idx[:total], d2[:total]

    def sphere_gather(self, center, radius):
        """All points within `radius` of `center`, ascending original index (camera_sensor.cpp:133-145, LiDAR mode)."""
        c = (C.c_double * 3)(*[float(v) for v in center])
        cnt = C.c_int64(0)
        self._check(self._L.pc_sphere_gather(self._h, c, float(radius), L.PC_HOST, C.c_void_p(0), 0, C.byref(cnt)))
        out = np.empty(max(cnt.value, 1), dtype=np.int32)
        self._check(self._L.pc_sphere_gather(self._h, c, float(radius), L.PC_HOST, C.c_void_p(out.ctypes.data), cnt.value, C.byref(cnt)))
        return out[: cnt.value]

    def sample_batch(self, sampler: L.PcSampler, k, advance=True):
        """The next k samples of the planner's stream, generated on the device (float64 (k, 3)); the sampler's engine state is
        advanced past them (pc_sample_batch)."""
        out = np.empty((int(k), 3), dtype=np.float64)
        st = C.c_uint32(0)
        self._check(self._L.pc_sample_batch(self._h, C.byref(sampler), int(k), L.PC_HOST, C.c_void_p(out.ctypes.data), C.byref(st)))
        if advance:
            sampler.engine_state = st.value
        return out

    def expand_batch(self, nodes: "PointCloudIndex", node_coord, node_radius, node_valid, sampler: L.PcSampler, params: L.PcRadiusParams,
                     z_l, safety_margin, k, cap=None, advance=True):
        """One speculative batch of the expansion loop on the device (pc_expand_batch): k samples steered against the frozen
        node set, radiusSearch for the centres against THIS index; returns the candidates the loop would keep as a structured
        array (center float64 x3, radius float32, nearest int32), in sample order."""
        nc = np.ascontiguousarray(node_coord, dtype=np.float64)
        nr = np.ascontiguousarray(node_radius, dtype=np.float32)
        nv = np.ascontiguousarray(node_valid, dtype=np.uint8)
        ns = L.PcNodeSet(nc.shape[0], nc.ctypes.data, nr.ctypes.data, nv.ctypes.data)
        cap = int(k) if cap is None else int(cap)
        out = np.empty(max(cap, 1), dtype=np.dtype(L.PC_CANDIDATE_DTYPE))
        assert out.dtype.itemsize == 32
        cnt, st = C.c_int64(0), C.c_uint32(0)
        self._check(self._L.pc_expand_batch(self._h, nodes._h, C.byref(ns), C.byref(sampler), C.byref(params), float(z_l), float(safety_margin),
                                            int(k), C.c_void_p(out.ctypes.data), cap, C.byref(cnt), C.byref(st)))
        if advance:
            sampler.engine_state = st.value
        return out[: cnt.value]

    def clearance(self, traj_first_seg, seg_order, seg_T, seg_coef_off, coef, params: L.PcRadiusParams,
                  t_now=None, dt=0.02, horizon=2.0):
        """checkSafeTrajectory for a batch of piecewise Bezier trajectories (host arrays, CSR layout of
        synth.bezier_trajectories).  Returns (first_hit int32, min_radius float32, n_samples int32)."""
        first = np.ascontiguousarray(traj_first_seg, dtype=np.int32)
        n_traj = first.shape[0] - 1
        tn = np.zeros(n_traj) if t_now is None else np.ascontiguousarray(t_now, dtype=np.float64)
        # pc_traj records {int32 first_seg, int32 num_seg, double t_now} filled without a Python loop
        traj = np.zeros(max(n_traj, 1), dtype=np.dtype([("first_seg", "<i4"), ("num_seg", "<i4"), ("t_now", "<f8")]))
        assert traj.dtype.itemsize == C.sizeof(L.PcTraj)
        traj["first_seg"][:n_traj] = first[:-1]
        traj["num_seg"][:n_traj] = np.diff(first)
        traj["t_now"][:n_traj] = tn
        so = np.ascontiguousarray(seg_order, dtype=np.int32)
        sT = np.ascontiguousarray(seg_T, dtype=np.float64)
        sc = np.ascontiguousarray(seg_coef_off, dtype=np.int64)
        cf = np.ascontiguousarray(coef, dtype=np.float64)
        fh = np.empty(n_traj, np.int32); mr = np.empty(n_traj, np.float32); ns = np.empty(n_traj, np.int32)
        vp = lambda a: C.c_void_p(a.ctypes.data)
        self._check(self._L.pc_clearance_batch(self._h, C.c_void_p(traj.ctypes.data), n_traj, vp(so), vp(sT), vp(sc), so.shape[0],
                                               vp(cf), cf.shape[0], L.PC_HOST, float(dt), float(horizon), C.byref(params),
                                               vp(fh), vp(mr), vp(ns)))
        return fh, mr, ns


def shard_range(m, rank, n_ranks):
    """Contiguous slice of m units owned by `rank` (pc_shard_range)."""
    b, e = C.c_int64(0), C.c_int64(0)
    L.load().pc_shard_range(int(m), int(rank), int(n_ranks), C.byref(b), C.byref(e))
    return b.value, e.value
