// segment_kernels.cuh -- pc_segment_nearest_batch: the exact nearest cloud point to each line segment [a, b].
//
// d2(p) is the fp64 expression of the contract (pc_index.h, DESIGN.md §4.11), evaluated by pc_seg_exact_d2 in exactly that
// operation order; the answer is the smallest (d2, original index), with the optional bound d2 <= r2 of pc_knn_batch.
//
//   pc_segment_kernel   one WARP per segment: the frontier walk of the kNN kernels (pc_warp_walk, knn_kernels.cuh: seeds, then
//                       up to 32 frontier nodes a step, depth-first close to the frontier's capacity) with the k = 1 list of
//                       pc_knn_wlist.  The segment's geometry pc_seg_geo supplies the walk's node test and leaf scan, as
//                       pc_sweep_geo does for pc_sphere_sweep_kernel (sweep_kernels.cuh).
//
// Node test (pc_seg_box): a child is pruned only if no point of its box can have fp64 d2 <= the current best (or the bound).
// Such a point lies within rho = sqrt(thr) + tau of the segment, where thr >= best (1 + 2^-20) is the kNN walks' fp32
// threshold and tau = 2^-48 |b - a| + 2^-100 covers the cancellation in W - t D (DESIGN.md §4.11 derives the bound).  Two
// tests, both with every rounding directed outwards:
//   gap   squared gap between the child box and the segment's AABB (rounded down) > rho^2 (rounded up): pruned; the gap is
//         also the frontier's ordering key;
//   slab  the segment's parameter interval [0, 1], clipped against the box dilated by rho on each axis (entry rounded down,
//         exit rounded up, reciprocals of |b - a| enclosed from both sides): empty -> pruned.
// Leaf scan: every point of a passing leaf, over its own `cnt`, gets the fp64 evaluation (an fp32 point prefilter -- the node
// test on the box [p, p] -- measured 10 % slower on long unbounded segments and 1-2 % faster bounded; DESIGN.md §4.11).
#pragma once
#include "knn_kernels.cuh"
#include <type_traits>

#define PC_SEG_WARPS 4                  // warps per CTA (32 KB of frontier)
#define PC_SEG_TAU_REL 0x1p-48f         // tau = |b - a| * 2^-48 + 2^-100 (DESIGN.md §4.11: 3.001 * 2^-53 |b - a| suffices)
#define PC_SEG_TAU_ABS 0x1p-100f

struct pc_seg_dev {
    double r2;                          // bound on the fp64 d2 (inclusive), +inf when unbounded
    float bound_thr;                    // its fp32 filter (pc_knn_dev_of), +inf when unbounded
};

// one segment, as every lane of its warp holds it
struct pc_seg_geo {
    double ax, ay, az, bx, by, bz;      // the endpoints, widened
    double dx, dy, dz, l2;              // D = B - A and L2 of the contract
    float lo[3], hi[3];                 // the segment's AABB
    float a[3];                         // a, negated on the axes where b < a (there the segment runs towards +)
    float inv_lo[3], inv_hi[3];         // enclosure of 1 / |b - a| per axis (+inf both when b == a on that axis)
    uint32_t flip;                      // bit i: axis i negated
    float tau;                          // absolute term of the threshold (distance units)
    float rho, thr2;                    // current search radius (distance) and its square, both rounded up
};

// the contract's expression (pc_index.h), operation for operation; pc_exact_d2(p, A) at the endpoint branches
__device__ __forceinline__ double pc_seg_exact_d2(float px, float py, float pz, const pc_seg_geo &G)
{
    const double wx = __dsub_rn((double)px, G.ax), wy = __dsub_rn((double)py, G.ay), wz = __dsub_rn((double)pz, G.az);
    const double s = __dadd_rn(__dadd_rn(__dmul_rn(wx, G.dx), __dmul_rn(wy, G.dy)), __dmul_rn(wz, G.dz));
    if (s <= 0.0 || G.l2 == 0.0) return pc_exact_d2(px, py, pz, G.ax, G.ay, G.az);
    if (s >= G.l2) return pc_exact_d2(px, py, pz, G.bx, G.by, G.bz);
    const double t = __ddiv_rn(s, G.l2);
    const double ex = __dsub_rn(wx, __dmul_rn(t, G.dx)), ey = __dsub_rn(wy, __dmul_rn(t, G.dy)), ez = __dsub_rn(wz, __dmul_rn(t, G.dz));
    return __dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez));
}

// rho and rho^2 from the point threshold thr (fp32, inclusive), both rounded up
__device__ __forceinline__ void pc_seg_set_thr(float thr, pc_seg_geo &G)
{
    G.rho = __fadd_ru(__fsqrt_ru(thr), G.tau);
    G.thr2 = __fmul_ru(G.rho, G.rho);
}

// returns |b - a| rounded up
__device__ __forceinline__ float pc_seg_setup(const float *a, const float *b, pc_seg_geo &G)
{
    G.ax = a[0]; G.ay = a[1]; G.az = a[2];
    G.bx = b[0]; G.by = b[1]; G.bz = b[2];
    G.dx = __dsub_rn(G.bx, G.ax); G.dy = __dsub_rn(G.by, G.ay); G.dz = __dsub_rn(G.bz, G.az);
    G.l2 = __dadd_rn(__dadd_rn(__dmul_rn(G.dx, G.dx), __dmul_rn(G.dy, G.dy)), __dmul_rn(G.dz, G.dz));
    G.flip = 0u;
    float len2 = 0.f;                   // |b - a|^2, rounded up
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const bool f = b[i] < a[i];
        const float s = f ? b[i] : a[i], e = f ? a[i] : b[i];      // the axis runs from s to e >= s
        G.lo[i] = s; G.hi[i] = e;
        G.a[i] = f ? -a[i] : a[i];
        G.flip |= (f ? 1u : 0u) << i;
        const float dlo = __fsub_rd(e, s), dhi = __fsub_ru(e, s);  // e - s > 0 is at least 2^-149 (no flush to zero here)
        G.inv_lo[i] = s == e ? INFINITY : __frcp_rd(dhi);
        G.inv_hi[i] = s == e ? INFINITY : __frcp_ru(dlo);
        len2 = __fadd_ru(len2, __fmul_ru(dhi, dhi));
    }
    const float len = __fsqrt_ru(len2);
    G.tau = __fmaf_ru(len, PC_SEG_TAU_REL, PC_SEG_TAU_ABS);
    return len;
}

// The box [lo, hi] against the segment: g2 = the squared gap between the box and the segment's AABB, rounded down (a lower
// bound of the squared distance of any of its points); [t0, t1] clipped against the box dilated by rho on each axis (entry
// rounded down, exit rounded up).  t0 > t1: every point of the clipped stretch is more than rho from the box.
__device__ __forceinline__ void pc_seg_clip(float lx, float ly, float lz, float hx, float hy, float hz, const pc_seg_geo &G,
                                            float &g2, float &t0, float &t1)
{
    const float lo[3] = { lx, ly, lz }, hi[3] = { hx, hy, hz };
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const float g = fmaxf(fmaxf(__fsub_rd(lo[i], G.hi[i]), __fsub_rd(G.lo[i], hi[i])), 0.f);
        g2 = __fadd_rd(g2, __fmul_rd(g, g));
        const bool f = (G.flip >> i) & 1u;
        const float bl = f ? -hi[i] : lo[i], bh = f ? -lo[i] : hi[i];
        const float nl = __fsub_rd(__fsub_rd(bl, G.rho), G.a[i]);   // <= (dilated lo) - a
        const float nh = __fsub_ru(__fadd_ru(bh, G.rho), G.a[i]);   // >= (dilated hi) - a
        // entry <= nl / |D|, exit >= nh / |D| for every |D| in the enclosure; 0 * inf (NaN) drops out of fmaxf / fminf
        t0 = fmaxf(t0, __fmul_rd(nl, nl >= 0.f ? G.inv_lo[i] : G.inv_hi[i]));
        t1 = fminf(t1, __fmul_ru(nh, nh >= 0.f ? G.inv_hi[i] : G.inv_lo[i]));
    }
}

// Node test of the box [lo, hi]: INFINITY if the slab test of [0, 1] proves it farther than rho from the segment, else the
// squared gap g2 of pc_seg_clip.
__device__ __forceinline__ float pc_seg_box(float lx, float ly, float lz, float hx, float hy, float hz, const pc_seg_geo &G)
{
    float g2 = 0.f, t0 = 0.f, t1 = 1.f;
    pc_seg_clip(lx, ly, lz, hx, hy, hz, G, g2, t0, t1);
    return t0 <= t1 ? g2 : INFINITY;
}

// the segment's leaf evaluation: the list key d2, and whether the bound K.r2 keeps it
__device__ __forceinline__ bool pc_seg_leaf(float px, float py, float pz, const pc_knn_dev &K, const pc_seg_geo &G, double &e)
{
    e = pc_seg_exact_d2(px, py, pz, G);
    return e <= K.r2;
}

// The hooks of pc_warp_walk (knn_kernels.cuh) for pc_seg_geo and pc_sweep_geo (sweep_kernels.cuh).  Each geometry supplies,
// by overload: pc_seg_box (node test: the frontier key, INFINITY when pruned), pc_walk_lim (the key limit), pc_seg_leaf (list
// key of a point, and whether it counts) and pc_seg_set_thr (refresh after the list's threshold changed).  The templates are
// constrained to the segment geometries: unconstrained, they would tie with pc_point_geo's hooks.
template <class GEO>
using pc_if_seg_geo = typename std::enable_if<std::is_base_of<pc_seg_geo, GEO>::value, int>::type;

// the limit the frontier's keys are tested against: rho^2 (the gap is a squared distance)
__device__ __forceinline__ float pc_walk_lim(const pc_seg_geo &G, const pc_knn_wlist &) { return G.thr2; }

template <class GEO, pc_if_seg_geo<GEO> = 0>
__device__ __forceinline__ float2 pc_walk_keys(const pc_rec &rec, const GEO &G)
{
    return make_float2(pc_seg_box(rec.L[0], rec.L[2], rec.L[4], rec.H[0], rec.H[2], rec.H[4], G),
                       pc_seg_box(rec.L[1], rec.L[3], rec.L[5], rec.H[1], rec.H[3], rec.H[5], G));
}

// scan NL leaves per lane (cnt points each; 0 = none) and offer the survivors to the k = 1 list
template <int NL, class GEO, pc_if_seg_geo<GEO> = 0>
__device__ __forceinline__ void pc_walk_scan(const pc_tree &T, const uint32_t (&ref)[NL], const uint32_t (&cnt)[NL], int lane,
                                             const pc_knn_dev &K, GEO &G, pc_knn_wlist &W)
{
    float4 p[NL * PC_LEAF];
#pragma unroll
    for (int j = 0; j < NL * PC_LEAF; j++)
        p[j] = (uint32_t)(j % PC_LEAF) < cnt[j / PC_LEAF] ? __ldg(T.points + (ref[j / PC_LEAF] & ~PC_REF_LEAF) + (j % PC_LEAF))
                                                          : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < NL * PC_LEAF; j++) {
        bool have = (uint32_t)(j % PC_LEAF) < cnt[j / PC_LEAF];
        double e = 0.0;
        uint32_t id = 0u;
        if (have) {
            have = pc_seg_leaf(p[j].x, p[j].y, p[j].z, K, G, e);
            id = (uint32_t)__float_as_int(p[j].w);
        }
        const float before = W.thr;
        pc_knn_warp_insert(have, e, id, lane, K, W);
        if (W.thr != before) pc_seg_set_thr(W.thr, G);
    }
}

// Work items: segment t of the batch, or of the curve order of the ordering pass (perm / ordered, m_eff its count).
// a / b: the endpoint arrays, stride floats per row.
__global__ void __launch_bounds__(32 * PC_SEG_WARPS)
pc_segment_kernel(pc_tree T, pc_seg_dev S, const float *__restrict__ a_xyz, const float *__restrict__ b_xyz, int64_t m, int stride,
                  const uint32_t *__restrict__ perm, const float4 *__restrict__ ordered, const unsigned long long *__restrict__ m_eff,
                  int32_t *__restrict__ out_idx, float *__restrict__ out_d2)
{
    __shared__ uint2 s_front[PC_SEG_WARPS][PC_KNN_FRONT];       // (inner node, float bits of its squared gap)
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
            pc_seg_geo G;
            pc_seg_setup(av, bv, G);
            pc_seg_set_thr(W.thr, G);
            pc_warp_walk(T, K, s_front[w], lane, G, W);
        }
        if (lane == 0) {
            if (out_idx) out_idx[slot] = finite ? (int32_t)W.li : -1;
            if (out_d2) out_d2[slot] = finite ? (float)W.ld : __int_as_float(0x7fc00000);
        }
        __syncwarp();
    }
}

// midpoints (x, y, z, 0) of the segments: the keys of the ordering pass
__global__ void pc_seg_mid_kernel(const float *__restrict__ a_xyz, const float *__restrict__ b_xyz, int64_t m, int stride, float4 *__restrict__ mid)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
        const float *a = a_xyz + i * stride, *b = b_xyz + i * stride;
        mid[i] = make_float4(0.5f * a[0] + 0.5f * b[0], 0.5f * a[1] + 0.5f * b[1], 0.5f * a[2] + 0.5f * b[2], 0.f);
    }
}
