// field_kernels.cuh -- the truncated distance field of the cloud on a voxel lattice (pc_distance_field).
//
// Voxel (i, j, k) of the lattice has the float32 centre c_a = (float)(origin_a + ((double)i_a + 0.5) * voxel), every fp64
// operation rounded to nearest and never fused.  Its entry is the row pc_knn_batch(k = 1, max_range) returns for that centre:
// the nearest point under (fp64 d2, original index), idx -1 where no point is within the bound, and the distance
// __dsqrt_rn(d2) rounded once to float32 (+inf for idx -1).
//
// One WARP per brick of 4 x 4 x 4 voxels: the 64 centres are made in registers from the lattice and walked as one 64-query
// packet with pc_packet_traverse<2> (query_kernels.cuh), lane l holding the voxels (l & 3, (l >> 2) & 3, l >> 4) and the
// same two layers up.  A brick is the tightest packet a batch of 64 queries can form, so the call needs none of what a query
// batch needs before its packets exist -- no curve keys, no sort, no gather, no permutation of the outputs -- and no
// packet_split deferral: the deferral catches packets cut across a jump of the curve order, and a brick's queries lie within
// a cube of 3 voxels' edge by construction.  Lanes whose voxels lie beyond a partial brick at the lattice's edge pass thr < 0.
// Bricks go to warps in 2 x 2 x 2 super-bricks (the four warps of a CTA take one 2 x 2 x 1 half), so that the warps resident
// on an SM walk neighbouring bricks and share node records in L1.
//
// Exactness: the walk runs with thr = the bound's fp32 filter (pc_knn_dev_of's bound_thr, FLT_MAX unbounded) and returns the
// smallest (d2, index) among the points that filter keeps -- every point with d2 <= r2 among them.  The inclusion test of
// the contract, d2 <= r2 in fp64, is applied to that minimum: if it fails, no point is within the bound.
#pragma once
#include "query_kernels.cuh"

#define PC_FIELD_WARPS 4                // warps per CTA (= PC_QUERY_THREADS / 32)

struct pc_field_dev {
    double origin[3], voxel;
    int64_t nx, ny, nz;                 // voxels of this launch (nz: the layers [k0, k0 + nz) of the lattice)
    int64_t k0;                         // first layer: the centres use the lattice's own k, the outputs start at layer k0
    int64_t bx, by, bz;                 // bricks per axis of this launch
    int wx, wy, wz;                     // super-brick width in bricks per axis (2, or 1 along an axis of one brick)
    int64_t sbx, sby;                   // super-bricks along x and y
    int64_t n_slots;                    // super-bricks x wx wy wz: warps the launch covers
    double r2;                          // bound on the fp64 d2 (inclusive), +inf when unbounded
    float bound_thr;                    // fp32 filter of the bound, FLT_MAX when unbounded
};

// the contract's centre coordinate of voxel i along one axis
__device__ __forceinline__ float pc_field_centre(double origin, double voxel, int64_t i)
{
    return __double2float_rn(__dadd_rn(origin, __dmul_rn(__dadd_rn((double)i, 0.5), voxel)));
}

__global__ void __launch_bounds__(PC_QUERY_THREADS, PC_PACKET_MIN_CTAS)
pc_distance_field_kernel(pc_tree T, pc_field_dev F, float *__restrict__ out_dist, int32_t *__restrict__ out_idx)
{
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = (int64_t)gridDim.x * PC_FIELD_WARPS;
    const int ws = F.wx * F.wy * F.wz;
    for (int64_t slot = (int64_t)blockIdx.x * PC_FIELD_WARPS + (threadIdx.x >> 5); slot < F.n_slots; slot += n_warps) {
        // slot -> super-brick (x fastest) and brick inside it (x, y, z bits: Morton order for 2 x 2 x 2)
        const int64_t sb = slot / ws;
        const int o = (int)(slot - sb * ws);
        const int64_t brx = (sb % F.sbx) * F.wx + o % F.wx;
        const int64_t bry = ((sb / F.sbx) % F.sby) * F.wy + (o / F.wx) % F.wy;
        const int64_t brz = (sb / (F.sbx * F.sby)) * F.wz + o / (F.wx * F.wy);
        if (brx >= F.bx || bry >= F.by || brz >= F.bz) continue;          // warp-uniform
        const int64_t i = brx * 4 + (lane & 3), j = bry * 4 + ((lane >> 2) & 3);
        float qv[2][3];
        pc_best b[2];
        bool valid[2];
        const float cx = pc_field_centre(F.origin[0], F.voxel, i < F.nx ? i : F.nx - 1);
        const float cy = pc_field_centre(F.origin[1], F.voxel, j < F.ny ? j : F.ny - 1);
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int64_t k = brz * 4 + 2 * h + (lane >> 4);
            valid[h] = i < F.nx && j < F.ny && k < F.nz;
            qv[h][0] = cx; qv[h][1] = cy;
            qv[h][2] = pc_field_centre(F.origin[2], F.voxel, F.k0 + (k < F.nz ? k : F.nz - 1));
            b[h].d2 = INFINITY; b[h].idx = -1;
            b[h].thr = (valid[h] && T.n_points > 0) ? F.bound_thr : -1.0f;     // thr < 0: this voxel needs nothing
        }
        pc_packet_traverse<2>(T, qv, b, lane);
#pragma unroll
        for (int h = 0; h < 2; h++) {
            if (!valid[h]) continue;
            const int64_t k = brz * 4 + 2 * h + (lane >> 4);
            const size_t v = (size_t)(i + F.nx * (j + F.ny * k));
            const bool hit = b[h].idx >= 0 && b[h].d2 <= F.r2;
            if (out_idx) out_idx[v] = hit ? b[h].idx : -1;
            if (out_dist) out_dist[v] = hit ? __double2float_rn(__dsqrt_rn(b[h].d2)) : INFINITY;
        }
    }
}
