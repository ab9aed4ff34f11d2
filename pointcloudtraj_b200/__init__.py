"""pointcloudtraj_b200 -- B200-native exact nearest-obstacle queries for pointcloudTraj's hot path.

The product is ``libpcindex.so`` (hand-written sm_100a CUDA behind the C ABI of ``include/pc_index.h``);
this package is the thin host-side mirror used by tests and bench.  It never imports ``oracle``.
"""
from ._lib import (PC_ARITH_FP64, PC_ARITH_PCL_FLOAT, PC_DEVICE, PC_HOST, PC_KNN_LARGE_MAX, PC_KNN_MAX, PC_QUERY_AUTO, PC_QUERY_SORTED, PC_QUERY_UNSORTED,  # noqa: F401
                   PC_RADIUS_BOUNDED, PC_RADIUS_FULL_NN, PcError, PcLattice, PcRadiusParams, PcSampler)
from .index import PointCloudIndex, shard_range  # noqa: F401

__all__ = ["PointCloudIndex", "PcRadiusParams", "PcSampler", "PcLattice", "PcError", "shard_range"]
