"""ctypes loader for libpcindex.so (the C ABI declared in include/pc_index.h).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no CPU
fallback: a missing library or a missing GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpcindex.so")

PC_OK, PC_EINVAL, PC_ENOMEM, PC_ECUDA, PC_ECAP, PC_ENCCL, PC_ENOTIMPL = 0, -1, -2, -3, -4, -5, -6
PC_HOST, PC_DEVICE, PC_HOST_ASYNC, PC_DEVICE_ASYNC = 0, 1, 2, 3
PC_RADIUS_BOUNDED, PC_RADIUS_FULL_NN = 0, 1
PC_QUERY_AUTO, PC_QUERY_UNSORTED, PC_QUERY_SORTED = 0, 2, 4
PC_ARITH_FP64, PC_ARITH_PCL_FLOAT = 0, 1
PC_NCCL_UNIQUE_ID_BYTES = 128
PC_KNN_MAX = 32
PC_KNN_LARGE_MAX = 1024

ERROR_NAMES = {PC_EINVAL: "PC_EINVAL", PC_ENOMEM: "PC_ENOMEM", PC_ECUDA: "PC_ECUDA", PC_ECAP: "PC_ECAP",
               PC_ENCCL: "PC_ENCCL", PC_ENOTIMPL: "PC_ENOTIMPL"}

# every symbol include/pc_index.h declares (tests/test_abi.py checks the library exports all of them)
ABI_SYMBOLS = [
    "pc_index_create", "pc_index_destroy", "pc_index_sync", "pc_last_error", "pc_version",
    "pc_index_build", "pc_index_size", "pc_index_view_get", "pc_index_last_build_ms",
    "pc_nearest_batch", "pc_radius_batch", "pc_range_batch", "pc_clearance_batch", "pc_sphere_gather",
    "pc_host_alloc", "pc_host_free",
    "pc_comm_unique_id", "pc_comm_init", "pc_comm_destroy", "pc_index_broadcast", "pc_shard_range",
    "pc_launch_count", "pc_profile_enable", "pc_profile_last_batch", "pc_batch_shard", "pc_index_set_radius_arith",
    "pc_profile_last_order_detail", "pc_profile_last_deferred_packets", "pc_sample_batch", "pc_expand_batch",
    "pc_knn_batch", "pc_range_sorted_batch", "pc_knn_large_batch", "pc_segment_nearest_batch", "pc_sphere_sweep_batch",
    "pc_trajectory_sweep_batch", "pc_trajectory_nearest_batch", "pc_distance_field",
]


class PcRadiusParams(C.Structure):
    """pc_radius_params: safeRegionRrtStar::setParam (Planner/src/corridor_finder.cpp:17-23) + start_pt (:43-50)."""
    _fields_ = [("search_margin", C.c_double), ("max_radius", C.c_double),
                ("sample_range", C.c_double), ("start", C.c_double * 3)]

    @classmethod
    def make(cls, search_margin=0.25, max_radius=1.5, sample_range=30.0, start=(0.0, 0.0, 0.0)):
        p = cls()
        p.search_margin, p.max_radius, p.sample_range = float(search_margin), float(max_radius), float(sample_range)
        p.start[0], p.start[1], p.start[2] = [float(v) for v in start]
        return p


class PcSampler(C.Structure):
    """pc_sampler: genSample's state while no path is known (corridor_finder.cpp:333-358) -- the minstd_rand0 engine state and
    the bounds setPt (:52-91) gives the uniform distributions."""
    _fields_ = [("engine_state", C.c_uint32), ("reserved", C.c_uint32), ("goal_ratio", C.c_double), ("inlier_ratio", C.c_double),
                ("end_pt", C.c_double * 3), ("lo", C.c_double * 3), ("hi", C.c_double * 3), ("in_lo", C.c_double * 3), ("in_hi", C.c_double * 3)]

    @classmethod
    def make(cls, start, end, box, sample_range, safety_margin, inlier_ratio, goal_ratio, engine_state=1):
        """The state after setParam(safety_margin, ., ., sample_range) + setPt(start, end, *box, ...); default_random_engine(0)
        starts from state 1."""
        s = cls()
        s.engine_state, s.goal_ratio, s.inlier_ratio = int(engine_state), float(goal_ratio), float(inlier_ratio)
        xl, xh, yl, yh, zl, zh = [float(v) for v in box]
        for a in range(3):
            s.end_pt[a] = float(end[a])
        s.lo[0], s.hi[0], s.lo[1], s.hi[1], s.lo[2], s.hi[2] = xl, xh, yl, yh, zl + safety_margin, zh
        s.in_lo[0], s.in_hi[0] = start[0] - sample_range, start[0] + sample_range
        s.in_lo[1], s.in_hi[1] = start[1] - sample_range, start[1] + sample_range
        s.in_lo[2], s.in_hi[2] = zl + safety_margin, zh
        return s


class PcNodeSet(C.Structure):
    _fields_ = [("n", C.c_int64), ("coord", C.c_void_p), ("radius", C.c_void_p), ("valid", C.c_void_p)]


PC_CANDIDATE_DTYPE = [("center", "<f8", (3,)), ("radius", "<f4"), ("nearest", "<i4")]      # pc_candidate, 32 bytes


class PcTraj(C.Structure):
    _fields_ = [("first_seg", C.c_int32), ("num_seg", C.c_int32), ("t_now", C.c_double)]


class PcLattice(C.Structure):
    """pc_lattice: nx x ny x nz voxels of edge `voxel`, the outer corner of voxel (0, 0, 0) at origin."""
    _fields_ = [("origin", C.c_double * 3), ("voxel", C.c_double), ("dims", C.c_int64 * 3)]

    @classmethod
    def make(cls, origin, voxel, dims):
        lat = cls()
        for a in range(3):
            lat.origin[a], lat.dims[a] = float(origin[a]), int(dims[a])
        lat.voxel = float(voxel)
        return lat


class PcIndexView(C.Structure):
    _fields_ = [("n_points", C.c_int64), ("n_nodes", C.c_int64), ("root", C.c_uint32), ("root_count", C.c_uint32),
                ("points", C.c_void_p), ("records", C.c_void_p),
                ("bbox_lo", C.c_float * 3), ("bbox_hi", C.c_float * 3)]


class PcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {msg}")
        self.code = code


_lib = None


def load():
    """Load libpcindex.so and declare the prototypes.  Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  pointcloudtraj_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int
    L.pc_index_create.argtypes = [C.POINTER(vp), i32, i64, vp]
    L.pc_index_destroy.argtypes = [vp]
    L.pc_index_destroy.restype = None
    L.pc_index_sync.argtypes = [vp]
    L.pc_last_error.argtypes = [vp]
    L.pc_last_error.restype = C.c_char_p
    L.pc_version.restype = C.c_char_p
    L.pc_index_build.argtypes = [vp, vp, i64, i64, i32]
    L.pc_index_size.argtypes = [vp]
    L.pc_index_size.restype = i64
    L.pc_index_view_get.argtypes = [vp, C.POINTER(PcIndexView)]
    L.pc_index_last_build_ms.argtypes = [vp, C.POINTER(C.c_float)]
    L.pc_nearest_batch.argtypes = [vp, vp, i64, i64, i32, i32, vp, vp]
    L.pc_knn_batch.argtypes = [vp, vp, i64, i64, i32, i32, i32, C.c_double, vp, vp]
    L.pc_knn_large_batch.argtypes = [vp, vp, i64, i64, i32, i32, i32, C.c_double, vp, vp]
    L.pc_segment_nearest_batch.argtypes = [vp, vp, vp, i64, i64, i32, i32, C.c_double, vp, vp]
    L.pc_sphere_sweep_batch.argtypes = [vp, vp, vp, i64, i64, i32, i32, C.c_double, vp, vp]
    L.pc_radius_batch.argtypes = [vp, vp, i64, i64, i32, i32, C.POINTER(PcRadiusParams), vp, vp]
    L.pc_range_batch.argtypes = [vp, vp, i64, i64, i32, vp, i32, vp, vp, i64]
    L.pc_range_sorted_batch.argtypes = [vp, vp, i64, i64, i32, vp, i32, i64, vp, vp, vp, i64]
    L.pc_clearance_batch.argtypes = [vp, vp, i64, vp, vp, vp, i64, vp, i64, i32, C.c_double, C.c_double,
                                     C.POINTER(PcRadiusParams), vp, vp, vp]
    L.pc_trajectory_sweep_batch.argtypes = [vp, vp, i64, vp, vp, vp, i64, vp, i64, i32, C.c_double, C.c_double, C.c_double,
                                            vp, vp, vp]
    L.pc_trajectory_nearest_batch.argtypes = [vp, vp, i64, vp, vp, vp, i64, vp, i64, i32, C.c_double, C.c_double, C.c_double,
                                              vp, vp, vp, vp]
    L.pc_distance_field.argtypes = [vp, C.POINTER(PcLattice), C.c_double, i32, vp, vp]
    L.pc_sphere_gather.argtypes = [vp, C.POINTER(C.c_double), C.c_double, i32, vp, i64, C.POINTER(i64)]
    L.pc_host_alloc.argtypes = [i64]
    L.pc_host_alloc.restype = vp
    L.pc_host_free.argtypes = [vp]
    L.pc_host_free.restype = None
    L.pc_comm_unique_id.argtypes = [C.c_char_p]
    L.pc_comm_init.argtypes = [C.POINTER(vp), i32, i32, C.c_char_p, i32]
    L.pc_comm_destroy.argtypes = [vp]
    L.pc_comm_destroy.restype = None
    L.pc_index_broadcast.argtypes = [vp, vp, i32]
    L.pc_shard_range.argtypes = [i64, i32, i32, C.POINTER(i64), C.POINTER(i64)]
    L.pc_shard_range.restype = None
    L.pc_launch_count.argtypes = [vp, i32]
    L.pc_launch_count.restype = i64
    L.pc_batch_shard.argtypes = [vp, i32, i32]
    L.pc_index_set_radius_arith.argtypes = [vp, i32]
    L.pc_profile_enable.argtypes = [vp, i32]
    L.pc_profile_last_batch.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.pc_profile_last_order_detail.argtypes = [vp, C.POINTER(C.c_float)]
    L.pc_profile_last_deferred_packets.argtypes = [vp, C.POINTER(C.c_int64)]
    L.pc_sample_batch.argtypes = [vp, C.POINTER(PcSampler), i64, i32, vp, C.POINTER(C.c_uint32)]
    L.pc_expand_batch.argtypes = [vp, vp, C.POINTER(PcNodeSet), C.POINTER(PcSampler), C.POINTER(PcRadiusParams), C.c_double, C.c_double,
                                  i64, vp, i64, C.POINTER(i64), C.POINTER(C.c_uint32)]
    _lib = L
    return L
