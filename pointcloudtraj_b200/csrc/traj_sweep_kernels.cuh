// traj_sweep_kernels.cuh -- pc_trajectory_sweep_batch: the certified first contact of a sphere of radius r moved along
// piecewise Bezier trajectories (contract in pc_index.h, DESIGN.md §4.13).
//
//   pc_traj_sweep_kernel  one WARP per trajectory.  The warp finds the trajectory's motion (the start of pc_clearance_batch,
//                         then the following segments up to the horizon), restricts each segment's control polygon to the
//                         motion with fp64 de Casteljau, and visits dyadic pieces [k / 2^d, (k + 1) / 2^d] of it earliest
//                         first -- (d, k) is the whole state, no stack:
//                           chord A = Q_0, B = Q_n of the piece's polygon; delta = the largest distance of a control point
//                           from the chord (the curve lies within delta of it, convex hull); the bounded nearest walk of
//                           pc_segment_kernel (pc_warp_walk, k = 1 list) around the chord at R = r + delta + mu;
//                           nothing within R: the piece is safe, go to the next one (coarsening while k is even);
//                           a point within R and sqrt(d2) + |B - A| + 2 mu <= r + tol: report the piece's start;
//                           otherwise split the piece (d + 1, 2k); at depth PC_TSW_DEPTH report the piece's start.
// mu = 2^-40 ((n + 1) S + r), S the largest |T c_j| of the segment, bounds every fp64 rounding of the polygons, the chord
// distance and the split parameters (DESIGN.md §4.13 derives it); the walk's fp32 node test is widened by the distance
// between the fp64 chord and its float32 copy, so it never prunes a point the fp64 leaf test would accept.
#pragma once
#include "segment_kernels.cuh"
#include "clearance_kernels.cuh"

#define PC_TSW_WARPS 4                  // warps per CTA (32 KB of frontier)
#define PC_TSW_DEPTH 50                 // subdivision depth cap: every call terminates
#define PC_TSW_MU_REL 0x1p-40           // mu = 2^-40 ((n + 1) S + r)  (DESIGN.md §4.13: about 2^-46 n S is needed)
#define PC_TSW_MAX_COORD 1e37           // control points beyond this magnitude count as non-finite (float32 chords)

// de Casteljau at t, in place: q[0..n] becomes the control polygon of the part [t, 1]
__device__ __forceinline__ void pc_dc_right(double (&q)[PC_MAX_ORDER + 1], int n, double t)
{
#pragma unroll
    for (int l = 1; l <= PC_MAX_ORDER; l++)
#pragma unroll
        for (int j = 0; j + l <= PC_MAX_ORDER; j++)
            if (j + l <= n) q[j] = __fma_rn(t, __dsub_rn(q[j + 1], q[j]), q[j]);
}

// de Casteljau at t, in place: q[0..n] becomes the control polygon of the part [0, t]
__device__ __forceinline__ void pc_dc_left(double (&q)[PC_MAX_ORDER + 1], int n, double t)
{
#pragma unroll
    for (int l = 1; l <= PC_MAX_ORDER; l++)
#pragma unroll
        for (int j = PC_MAX_ORDER; j >= l; j--)
            if (j <= n) q[j] = __fma_rn(t, __dsub_rn(q[j], q[j - 1]), q[j - 1]);
}

// squared distance of P from the segment A + t D, t in [0, 1] (fp64; its rounding is part of mu)
__device__ __forceinline__ double pc_tsw_d2(double px, double py, double pz, double ax, double ay, double az,
                                            double dx, double dy, double dz, double l2)
{
    double wx = px - ax, wy = py - ay, wz = pz - az;
    const double s = wx * dx + wy * dy + wz * dz;
    if (s > 0.0 && l2 > 0.0) {
        const double t = s >= l2 ? 1.0 : s / l2;
        wx -= t * dx; wy -= t * dy; wz -= t * dz;
    }
    return wx * wx + wy * wy + wz * wz;
}

__device__ __forceinline__ double pc_warp_dmax(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(PC_FULL_MASK, v, o));
    return v;
}

// The parts of a trajectory walk that pc_traj_sweep_kernel and pc_traj_nearest_kernel (traj_nearest_kernels.cuh) share.
// The motion of one trajectory: segments i0 .. last (indices into the trajectory), local times [t_s, T] on the first, [0, T]
// between, [0, s_end] on the last; finite: every segment of it has a usable T, order and coefficients.
struct pc_traj_motion {
    int i0, last;                       // last = -1: empty motion
    double t_s, s_end;
    bool finite;
};

// the motion of trajectory tj up to `horizon` (called by the whole warp: the finiteness check is spread over the lanes)
__device__ __forceinline__ pc_traj_motion pc_traj_motion_of(const pc_traj_dev &tj, const int32_t *__restrict__ seg_order,
                                                            const double *__restrict__ seg_T, const int64_t *__restrict__ seg_coef_off,
                                                            const double *__restrict__ coef, double horizon, int lane)
{
    const int32_t seg0 = tj.first_seg, nseg = tj.num_seg;
    pc_traj_motion m;
    // the start of pc_clearance_kernel (sim_planning_demo.cpp:735-742): segment seg0 + i0, local time t_s
    int i0 = 0;
    double t_s = tj.t_now > 0.0 ? tj.t_now : 0.0;
    for (i0 = 0; i0 < nseg; ++i0) {
        if (t_s > seg_T[seg0 + i0] && i0 + 1 < nseg) t_s = __dsub_rn(t_s, seg_T[seg0 + i0]);
        else break;
    }
    // the time left (rem) and s_end are rounded up: the motion is never cut short
    int last = -1;
    double s_end = 0.0;
    bool finite = true;
    if (nseg > 0 && horizon >= 0.0 && !(t_s > seg_T[seg0 + i0])) {
        double rem = horizon;
        for (int j = i0; j < nseg; j++) {
            const int32_t s = seg0 + j;
            const double Ts = seg_T[s];
            const int n = seg_order[s];
            bool ok = Ts > 0.0 && Ts < INFINITY && n >= 1 && n <= PC_MAX_ORDER;
            if (ok) {
                const double *c = coef + seg_coef_off[s];
                bool bad = false;
                for (int e = lane; e < 3 * (n + 1); e += 32) bad = bad || !(fabs(__dmul_rn(Ts, c[e])) <= PC_TSW_MAX_COORD);
                ok = !__any_sync(PC_FULL_MASK, bad);
            }
            finite = finite && ok;
            last = j;
            const double sa = j == i0 ? t_s : 0.0;
            const double e = __dadd_ru(sa, rem);
            if (e < Ts) { s_end = e; break; }
            s_end = Ts;
            rem = __dsub_ru(rem, __dsub_rd(Ts, sa));
            if (!(rem >= 0.0)) break;
        }
    }
    m.i0 = i0; m.last = last; m.t_s = t_s; m.s_end = s_end; m.finite = finite;
    return m;
}

// The control polygon T c_j (order n, coefficients c) restricted to the local times [sa, sb] of the motion, into M (lanes
// 0..2, one axis each).  The motion's part in u = sigma / T is [ua, ub] rounded outwards; the restriction splits at ua, then
// at t2 rounded down, so that it ends at or before ub (DESIGN.md §4.13: the sliver is inside mu).  Returns
// mu = 2^-40 ((n + 1) S + radius); ua and span (<= the restriction's length in u) place a piece's start in time.
__device__ __forceinline__ double pc_traj_restrict(const double *__restrict__ c, double Ts, int n, double sa, double sb, double radius,
                                                   int lane, double (*M)[PC_MAX_ORDER + 1], double &ua, double &span)
{
    const int nc = n + 1;
    ua = __ddiv_rd(sa, Ts);
    const double ub = fmin(1.0, __ddiv_ru(sb, Ts));
    const double t2 = (ub > ua && ua < 1.0) ? fmin(1.0, __ddiv_rd(__dsub_rd(ub, ua), __dsub_ru(1.0, ua))) : 0.0;
    span = __dmul_rd(t2, __dsub_rd(1.0, ua));
    double s2 = 0.0;
    if (lane < nc) {
        const double x = __dmul_rn(Ts, c[lane]), y = __dmul_rn(Ts, c[nc + lane]), z = __dmul_rn(Ts, c[2 * nc + lane]);
        s2 = x * x + y * y + z * z;
    }
    const double mu = PC_TSW_MU_REL * ((double)nc * sqrt(pc_warp_dmax(s2)) + radius);
    if (lane < 3) {
        double q[PC_MAX_ORDER + 1];
#pragma unroll
        for (int i = 0; i <= PC_MAX_ORDER; i++) q[i] = i <= n ? __dmul_rn(Ts, c[lane * nc + i]) : 0.0;
        pc_dc_right(q, n, ua);
        pc_dc_left(q, n, t2);
#pragma unroll
        for (int i = 0; i <= PC_MAX_ORDER; i++) if (i <= n) M[lane][i] = q[i];
    }
    __syncwarp();
    return mu;
}

// One piece [k / 2^d, (k + 1) / 2^d] of the restricted polygon M, into Q: its chord A = Q_0, B = Q_n, |B - A|^2 (l2) and
// delta, the largest fp64 distance of a control point from the chord (the piece of the curve lies within delta of it).
struct pc_traj_chord {
    double ax, ay, az, bx, by, bz, l2, delta;
};

__device__ __forceinline__ pc_traj_chord pc_traj_piece(const double (*M)[PC_MAX_ORDER + 1], double (*Q)[PC_MAX_ORDER + 1], int n,
                                                       unsigned long long k, int d, double a, int lane)
{
    const int nc = n + 1;
    if (lane < 3) {
        double q[PC_MAX_ORDER + 1];
#pragma unroll
        for (int i = 0; i <= PC_MAX_ORDER; i++) q[i] = i <= n ? M[lane][i] : 0.0;
        pc_dc_right(q, n, a);
        pc_dc_left(q, n, __ddiv_rn(1.0, (double)((1ull << d) - k)));    // (b - a) / (1 - a)
#pragma unroll
        for (int i = 0; i <= PC_MAX_ORDER; i++) if (i <= n) Q[lane][i] = q[i];
    }
    __syncwarp();
    pc_traj_chord C;
    C.ax = Q[0][0]; C.ay = Q[1][0]; C.az = Q[2][0];
    const double dx = Q[0][n] - C.ax, dy = Q[1][n] - C.ay, dz = Q[2][n] - C.az;
    C.l2 = dx * dx + dy * dy + dz * dz;
    double dev = 0.0;
    if (lane < nc) dev = pc_tsw_d2(Q[0][lane], Q[1][lane], Q[2][lane], C.ax, C.ay, C.az, dx, dy, dz, C.l2);
    C.delta = sqrt(pc_warp_dmax(dev));
    C.bx = Q[0][n]; C.by = Q[1][n]; C.bz = Q[2][n];
    __syncwarp();                                   // Q is read before lanes 0..2 write the next piece
    return C;
}

// The nearest cloud point to the fp64 chord within R (R = +inf: unbounded): pc_segment_kernel's walk with the k = 1 list.
// W.ki == PC_KNN_NONE: no point within R; else W.kd is its fp64 squared distance from the chord.  The node test runs on the
// float32 chord, widened by its distance from the fp64 chord of the leaf test, so it never prunes a point the leaf test keeps.
__device__ __forceinline__ void pc_traj_chord_walk(const pc_tree &T, uint2 *__restrict__ F, int lane, const pc_traj_chord &C,
                                                   double R, pc_knn_wlist &W)
{
    const double r2 = __dmul_ru(R, R);
    const pc_knn_dev K = pc_knn_dev_k1(r2, pc_thr_from(r2));
    W = pc_knn_wlist_empty(K.bound_thr);
    if (T.n_points > 0) {
        const double ax = C.ax, ay = C.ay, az = C.az, bx = C.bx, by = C.by, bz = C.bz;
        const float af[3] = { (float)ax, (float)ay, (float)az }, bf[3] = { (float)bx, (float)by, (float)bz };
        pc_seg_geo G;
        pc_seg_setup(af, bf, G);
        G.ax = ax; G.ay = ay; G.az = az; G.bx = bx; G.by = by; G.bz = bz;
        G.dx = __dsub_rn(bx, ax); G.dy = __dsub_rn(by, ay); G.dz = __dsub_rn(bz, az);
        G.l2 = __dadd_rn(__dadd_rn(__dmul_rn(G.dx, G.dx), __dmul_rn(G.dy, G.dy)), __dmul_rn(G.dz, G.dz));
        const double ea = pc_exact_d2(af[0], af[1], af[2], ax, ay, az), eb = pc_exact_d2(bf[0], bf[1], bf[2], bx, by, bz);
        const float ef = __double2float_ru(1.0000001 * sqrt(fmax(ea, eb)));
        G.tau = __fadd_ru(G.tau, ef);
        pc_seg_set_thr(W.thr, G);
        pc_warp_walk(T, K, F, lane, G, W);
    }
}

// Outputs per trajectory (each nullable): the contact's segment (index into the segment arrays), its local time rounded so
// that nothing before it touches, and the witness point's original index; -1 / +inf / -1 without contact, -1 / NaN / -1
// when a segment of the motion has a non-finite (or unusable) T, order or coefficient.
__global__ void __launch_bounds__(32 * PC_TSW_WARPS)
pc_traj_sweep_kernel(pc_tree T, const pc_traj_dev *__restrict__ traj, int64_t n_traj, const int32_t *__restrict__ seg_order,
                     const double *__restrict__ seg_T, const int64_t *__restrict__ seg_coef_off, const double *__restrict__ coef,
                     double horizon, double radius, double tol,
                     int32_t *__restrict__ out_seg, double *__restrict__ out_s, int32_t *__restrict__ out_idx)
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
        int32_t res_seg = -1, res_idx = -1;
        double res_s = mo.finite ? INFINITY : __longlong_as_double(0x7ff8000000000000ll);
        for (int j = mo.i0; mo.finite && j <= mo.last; j++) {
            const int32_t s = seg0 + j;
            const double Ts = seg_T[s];
            const int n = seg_order[s];
            const double *c = coef + seg_coef_off[s];
            const double sa = j == mo.i0 ? mo.t_s : 0.0, sb = j == mo.last ? mo.s_end : Ts;
            double ua, span;
            const double mu = pc_traj_restrict(c, Ts, n, sa, sb, radius, lane, M, ua, span);
            unsigned long long k = 0ull;
            int d = 0;
            for (;;) {
                const double a = ldexp((double)k, -d);                             // exact
                const pc_traj_chord C = pc_traj_piece(M, Q, n, k, d, a, lane);
                const double R = __dadd_ru(__dadd_ru(radius, C.delta), mu);
                pc_knn_wlist W;
                pc_traj_chord_walk(T, s_front[w], lane, C, R, W);
                if (W.ki == PC_KNN_NONE) {                      // safe: the next piece, as coarse as the order allows
                    k++;
                    while (d > 0 && !(k & 1ull)) { k >>= 1; d--; }
                    if (d == 0) break;
                    continue;
                }
                const double reach = __dadd_ru(__dadd_ru(__dsqrt_ru(W.kd), __dsqrt_ru(C.l2)), 2.0 * mu);
                if (reach <= __dadd_rd(radius, tol) || d == PC_TSW_DEPTH) {
                    res_seg = s;
                    res_idx = (int32_t)W.ki;
                    res_s = fmax(sa, __dmul_rd(Ts, __fma_rd(a, span, ua)));
                    break;
                }
                d++;
                k <<= 1;
            }
            if (res_seg >= 0) break;
        }
        if (lane == 0) {
            if (out_seg) out_seg[tr] = res_seg;
            if (out_s) out_s[tr] = res_s;
            if (out_idx) out_idx[tr] = res_idx;
        }
        __syncwarp();
    }
}
