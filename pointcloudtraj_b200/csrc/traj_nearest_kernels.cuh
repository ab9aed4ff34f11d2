// traj_nearest_kernels.cuh -- pc_trajectory_nearest_batch: the certified clearance of piecewise Bezier trajectories, i.e. the
// distance from the motion to the nearest cloud point to within tol, with a witness (contract in pc_index.h, DESIGN.md §4.14).
//
//   pc_traj_nearest_kernel  one WARP per trajectory.  The motion, the fp64 de Casteljau restriction of each segment, the
//                           dyadic pieces (d, k) and the chord walk are pc_traj_sweep_kernel's (traj_sweep_kernels.cuh); the
//                           search over the pieces is branch and bound on the distance instead of the earliest contact.
//                           U is the best upper bound so far (max_range + tol when bounded, +inf when not).  Per piece, with
//                           chord A, B, delta and the nearest point p to the chord at fp64 squared distance kd:
//                             no point within (U - tol + delta)(1 + 2^-40) + mu: pruned, every point of the piece is at
//                             least U - tol from the cloud;
//                             lb = sqrt(kd)(1 - 2^-40) - delta - mu <= the piece's distance from the cloud: lb >= U - tol
//                             prunes the piece;
//                             otherwise two upper bounds, each with its witness: ub = (sqrt(kd) + |B - A|)(1 + 2^-40) + mu
//                             >= |C(piece start) - p|, and the nearest point q to B (a point walk from B rounded to float)
//                             >= |C(piece end) - q|; below U they become U.  Then lb >= U - tol prunes the piece, otherwise
//                             it is split (at depth PC_TSW_DEPTH it is accepted).
//                           Once U - tol <= 0 nothing can improve the certificate and the trajectory ends.  Every walk is
//                           bounded, at most at PC_TNR_MAX_R: an unbounded one that never meets a finite point keeps an
//                           infinite frontier limit, and the walk's "no child" sentinel is an infinite key.
// mu = 2^-40 (n + 1) S (the sweep's mu without its radius term); the fp64 chord distance errs relative to the distance itself,
// which can be tens of metres unbounded, so that term is the separate factor 1 -/+ 2^-40 (DESIGN.md §4.14 derives both).
#pragma once
#include "traj_sweep_kernels.cuh"

#define PC_TNR_REL_UP (1.0 + 0x1p-40)      // the chord distance's relative error, widened (DESIGN.md §4.14: about 4 u is needed)
#define PC_TNR_REL_DN (1.0 - 0x1p-40)
#define PC_TNR_MAX_R 0x1p60                // the largest distance searched (its square and fp32 filter stay finite)

// The nearest cloud point q to B within U (at most PC_TNR_MAX_R), by the point walk of the kNN kernels from B rounded to
// float: returns ub >= |C - q| for the curve point C within mu of B, and q's original index (PC_KNN_NONE: none within U).
// Not inlined: a second walk inlined into the kernel spills.
__device__ __noinline__ double pc_tnr_point_bound(const pc_tree &T, uint2 *__restrict__ F, int lane, double bx, double by,
                                                  double bz, double U, double mu, uint32_t &qi)
{
    pc_point_geo P;
    P.qx = (float)bx; P.qy = (float)by; P.qz = (float)bz;
    const double eb = pc_exact_d2(P.qx, P.qy, P.qz, bx, by, bz);                 // |B - float(B)|^2
    const double Ur = fmin(U, PC_TNR_MAX_R);
    const double r2 = __dmul_ru(Ur, Ur);
    const pc_knn_dev K = pc_knn_dev_k1(r2, pc_thr_from(r2));
    pc_knn_wlist V = pc_knn_wlist_empty(K.bound_thr);
    pc_warp_walk(T, K, F, lane, P, V);
    qi = V.ki;
    return __dadd_ru(__dmul_ru(__dadd_ru(__dsqrt_ru(V.kd), __dsqrt_ru(eb)), PC_TNR_REL_UP), mu);
}

// Outputs per trajectory (each nullable): the witness's segment (index into the segment arrays), its local time, the witness
// point's original index and d >= |C(s, sigma) - p|, with nothing on the motion closer than d - tol to the cloud;
// -1 / +inf / -1 / +inf without a witness, -1 / NaN / -1 / NaN when a segment of the motion is not finite.
__global__ void __launch_bounds__(32 * PC_TSW_WARPS)
pc_traj_nearest_kernel(pc_tree T, const pc_traj_dev *__restrict__ traj, int64_t n_traj, const int32_t *__restrict__ seg_order,
                       const double *__restrict__ seg_T, const int64_t *__restrict__ seg_coef_off, const double *__restrict__ coef,
                       double horizon, double max_range, double tol,
                       int32_t *__restrict__ out_seg, double *__restrict__ out_s, int32_t *__restrict__ out_idx,
                       double *__restrict__ out_dist)
{
    __shared__ uint2 s_front[PC_TSW_WARPS][PC_KNN_FRONT];                      // (inner node, float bits of its squared gap)
    __shared__ double s_poly[PC_TSW_WARPS][2][3][PC_MAX_ORDER + 1];            // per axis: the segment on the motion, the piece
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    double (*M)[PC_MAX_ORDER + 1] = s_poly[w][0];
    double (*Q)[PC_MAX_ORDER + 1] = s_poly[w][1];
    for (int64_t tr = (int64_t)blockIdx.x * PC_TSW_WARPS + w; tr < n_traj; tr += (int64_t)gridDim.x * PC_TSW_WARPS) {
        const pc_traj_dev tj = traj[tr];
        const int32_t seg0 = tj.first_seg;
        const pc_traj_motion mo = pc_traj_motion_of(tj, seg_order, seg_T, seg_coef_off, coef, horizon, lane);
        double U = max_range >= 0.0 ? __dadd_ru(max_range, tol) : INFINITY;
        int32_t res_seg = -1, res_idx = -1;
        double res_s = mo.finite ? INFINITY : __longlong_as_double(0x7ff8000000000000ll);
        bool done = false;
        for (int j = mo.i0; mo.finite && !done && j <= mo.last; j++) {
            const int32_t s = seg0 + j;
            const double Ts = seg_T[s];
            const int n = seg_order[s];
            const double *c = coef + seg_coef_off[s];
            const double sa = j == mo.i0 ? mo.t_s : 0.0, sb = j == mo.last ? mo.s_end : Ts;
            double ua, span;
            const double mu = pc_traj_restrict(c, Ts, n, sa, sb, 0.0, lane, M, ua, span);
            unsigned long long k = 0ull;
            int d = 0;
            for (;;) {
                const double cut = __dsub_ru(U, tol);                               // >= U - tol; +inf unbounded
                if (!(cut > 0.0)) { done = true; break; }                           // d - tol <= 0 certifies itself
                const double a = ldexp((double)k, -d);                             // exact
                const pc_traj_chord C = pc_traj_piece(M, Q, n, k, d, a, lane);
                pc_knn_wlist W;
                const double R = __dadd_ru(__dmul_ru(__dadd_ru(cut, C.delta), PC_TNR_REL_UP), mu);
                pc_traj_chord_walk(T, s_front[w], lane, C, fmin(R, PC_TNR_MAX_R), W);
                bool next = W.ki == PC_KNN_NONE;
                if (!next) {
                    const double lb = __dsub_rd(__dsub_rd(__dmul_rd(__dsqrt_rd(W.kd), PC_TNR_REL_DN), C.delta), mu);
                    next = lb >= cut;
                    if (!next) {
                        const double ub = __dadd_ru(__dmul_ru(__dadd_ru(__dsqrt_ru(W.kd), __dsqrt_ru(C.l2)), PC_TNR_REL_UP), mu);
                        if (ub < U) {
                            U = ub;
                            res_seg = s;
                            res_idx = (int32_t)W.ki;
                            res_s = fmax(sa, __dmul_rd(Ts, __fma_rd(a, span, ua)));
                        }
                        // the piece end's nearest point: on a stretch that approaches the cloud it bounds the piece's
                        // distance within about delta, where the chord bound needs |B - A| <= tol
                        uint32_t qi;
                        const double ubq = pc_tnr_point_bound(T, s_front[w], lane, C.bx, C.by, C.bz, U, mu, qi);
                        if (qi != PC_KNN_NONE) {
                            if (ubq < U) {
                                U = ubq;
                                res_seg = s;
                                res_idx = (int32_t)qi;
                                res_s = fmax(sa, __dmul_rd(Ts, __fma_rd(ldexp((double)(k + 1ull), -d), span, ua)));
                            }
                        }
                        next = lb >= __dsub_ru(U, tol) || d == PC_TSW_DEPTH;
                    }
                }
                if (next) {                                     // decided: the next piece, as coarse as the order allows
                    k++;
                    while (d > 0 && !(k & 1ull)) { k >>= 1; d--; }
                    if (d == 0) break;
                    continue;
                }
                d++;
                k <<= 1;
            }
        }
        if (lane == 0) {
            if (out_seg) out_seg[tr] = res_seg;
            if (out_s) out_s[tr] = res_s;
            if (out_idx) out_idx[tr] = res_idx;
            if (out_dist) out_dist[tr] = res_seg >= 0 ? U : res_s;
        }
        __syncwarp();
    }
}
