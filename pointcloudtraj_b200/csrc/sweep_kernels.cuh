// sweep_kernels.cuh -- pc_sphere_sweep_batch: the first contact of a sphere of radius r swept from a to b with the cloud.
//
// t(p) is the fp64 expression of the contract (pc_index.h, DESIGN.md §4.12), evaluated by pc_sweep_exact_t in exactly that
// operation order; the answer is the smallest (t, original index).
//
//   pc_sphere_sweep_kernel  one WARP per segment: the walk of pc_segment_kernel (pc_warp_walk, knn_kernels.cuh) with
//                           t(p) as the key of the k = 1 list (pc_knn_wlist: (key, index) order, the lowest index on ties).
//
// Node test (pc_seg_box of pc_sweep_geo): a point with a computed contact at t lies within rho of the exact segment point
// A + t (B - A), where rho = r (rounded up) + 2^-20 (r + |b - a|) + 2^-100 is fixed per segment (DESIGN.md §4.12 derives the
// bound).  A child is pruned when its squared gap to the segment's AABB exceeds rho^2, or when the parameter interval
// [0, min(1, thr)] clipped against the box dilated by rho is empty; thr = pc_thr_from(best t) is the list's fp32 threshold,
// inclusive, so an exact tie at a lower index survives.  The clip's entry (rounded down) is the frontier's key.
#pragma once
#include "segment_kernels.cuh"

#define PC_SWEEP_RHO_REL 0x1p-20f       // rho = r + 2^-20 (r + |b - a|) + 2^-100 (DESIGN.md §4.12: 2^-23.2 (r + |b - a|) suffices)

// the segment's geometry, rho fixed, and the list's bound on t
struct pc_sweep_geo : pc_seg_geo {
    float tmax;                         // min(1, thr): a contact beyond it can neither beat nor tie the best
};

// the contract's expression (pc_index.h), operation for operation: t(p) in [0, 1], or INFINITY where p makes no contact
__device__ __forceinline__ double pc_sweep_exact_t(float px, float py, float pz, const pc_seg_geo &G, double r2)
{
    const double wx = __dsub_rn((double)px, G.ax), wy = __dsub_rn((double)py, G.ay), wz = __dsub_rn((double)pz, G.az);
    const double c0 = __dadd_rn(__dadd_rn(__dmul_rn(wx, wx), __dmul_rn(wy, wy)), __dmul_rn(wz, wz));  // pc_exact_d2(p, A)
    if (c0 <= r2) return 0.0;
    if (G.l2 != 0.0) {
        const double s = __dadd_rn(__dadd_rn(__dmul_rn(wx, G.dx), __dmul_rn(wy, G.dy)), __dmul_rn(wz, G.dz));
        if (s > 0.0) {
            const double h = __dsub_rn(c0, r2);
            const double disc = __dsub_rn(__dmul_rn(s, s), __dmul_rn(G.l2, h));
            if (disc >= 0.0) {
                const double t = __ddiv_rn(h, __dadd_rn(s, __dsqrt_rn(disc)));
                if (t <= 1.0) return t;
            }
        }
    }
    return pc_exact_d2(px, py, pz, G.bx, G.by, G.bz) <= r2 ? 1.0 : INFINITY;
}

// node test: INFINITY when pruned (gap above rho^2, or [0, tmax] clipped empty), else the clip's entry, rounded down
__device__ __forceinline__ float pc_seg_box(float lx, float ly, float lz, float hx, float hy, float hz, const pc_sweep_geo &G)
{
    float g2 = 0.f, t0 = 0.f, t1 = G.tmax;
    pc_seg_clip(lx, ly, lz, hx, hy, hz, G, g2, t0, t1);
    return t0 <= t1 && g2 <= G.thr2 ? t0 : INFINITY;
}

__device__ __forceinline__ float pc_walk_lim(const pc_sweep_geo &G, const pc_knn_wlist &) { return G.tmax; }

__device__ __forceinline__ bool pc_seg_leaf(float px, float py, float pz, const pc_knn_dev &K, const pc_sweep_geo &G, double &e)
{
    e = pc_sweep_exact_t(px, py, pz, G, K.r2);
    return e <= 1.0;
}

// rho stays fixed; only the bound on t follows the list
__device__ __forceinline__ void pc_seg_set_thr(float thr, pc_sweep_geo &G) { G.tmax = fminf(1.f, thr); }

// Work items as in pc_segment_kernel.  S.r2 = R2 of the contract, S.bound_thr = +inf; r_up = the radius rounded up to float.
__global__ void __launch_bounds__(32 * PC_SEG_WARPS)
pc_sphere_sweep_kernel(pc_tree T, pc_seg_dev S, float r_up, const float *__restrict__ a_xyz, const float *__restrict__ b_xyz,
                       int64_t m, int stride, const uint32_t *__restrict__ perm, const float4 *__restrict__ ordered,
                       const unsigned long long *__restrict__ m_eff, int32_t *__restrict__ out_idx, float *__restrict__ out_t)
{
    __shared__ uint2 s_front[PC_SEG_WARPS][PC_KNN_FRONT];       // (inner node, float bits of its entry parameter)
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const pc_knn_dev K = pc_knn_dev_k1(S.r2, S.bound_thr);
    const long long m_search = m_eff ? (long long)*m_eff : (long long)m;
    const long long n_warps = (long long)gridDim.x * PC_SEG_WARPS;
    for (long long t = (long long)blockIdx.x * PC_SEG_WARPS + w; t < m_search; t += n_warps) {
        const uint32_t slot = pc_query_fetch(perm, ordered, t);
        const float *a = a_xyz + (size_t)slot * stride, *b = b_xyz + (size_t)slot * stride;
        const float av[3] = { a[0], a[1], a[2] }, bv[3] = { b[0], b[1], b[2] };
        const bool finite = isfinite(av[0]) && isfinite(av[1]) && isfinite(av[2]) && isfinite(bv[0]) && isfinite(bv[1]) && isfinite(bv[2]);
        pc_knn_wlist W = pc_knn_wlist_empty(S.bound_thr);
        if (finite && T.n_points > 0) {
            pc_sweep_geo G;
            const float len = pc_seg_setup(av, bv, G);
            G.rho = __fadd_ru(r_up, __fmaf_ru(__fadd_ru(r_up, len), PC_SWEEP_RHO_REL, PC_SEG_TAU_ABS));
            G.thr2 = __fmul_ru(G.rho, G.rho);
            pc_seg_set_thr(W.thr, G);
            pc_warp_walk(T, K, s_front[w], lane, G, W);
        }
        if (lane == 0) {
            if (out_idx) out_idx[slot] = finite ? (int32_t)W.li : -1;
            if (out_t) out_t[slot] = finite ? __double2float_rd(W.ld) : __int_as_float(0x7fc00000);
        }
        __syncwarp();
    }
}
