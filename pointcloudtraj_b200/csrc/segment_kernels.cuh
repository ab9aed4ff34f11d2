// segment_kernels.cuh -- pc_segment_nearest_batch: the exact nearest cloud point to each line segment [a, b].
//
// d2(p) is the fp64 expression of the contract (pc_index.h, DESIGN.md §4.11), evaluated by pc_seg_exact_d2 in exactly that
// operation order; the answer is the smallest (d2, original index), with the optional bound d2 <= r2 of pc_knn_batch.
//
//   pc_segment_kernel   one WARP per segment: the frontier walk of pc_knn_warp_search (seeds, then up to 32 frontier nodes a
//                       step, depth-first close to the frontier's capacity) with the k = 1 list of pc_knn_wlist.  The walk is a
//                       copy, not an instantiation: the node test and the leaf scan differ, and the existing kNN kernels stay
//                       byte-identical.
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

__device__ __forceinline__ void pc_seg_setup(const float *a, const float *b, pc_seg_geo &G)
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
    G.tau = __fmaf_ru(__fsqrt_ru(len2), PC_SEG_TAU_REL, PC_SEG_TAU_ABS);
}

// Node test of the box [lo, hi]: INFINITY if the slab test proves it farther than rho from the segment, else the squared gap
// between the box and the segment's AABB, rounded down (a lower bound of the squared distance of any of its points).
__device__ __forceinline__ float pc_seg_box(float lx, float ly, float lz, float hx, float hy, float hz, const pc_seg_geo &G)
{
    const float lo[3] = { lx, ly, lz }, hi[3] = { hx, hy, hz };
    float g2 = 0.f, t0 = 0.f, t1 = 1.f;
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
    return t0 <= t1 ? g2 : INFINITY;
}

// scan NL leaves per lane (cnt points each; 0 = none) and offer the survivors to the k = 1 list
template <int NL>
__device__ __forceinline__ void pc_seg_scan(const pc_tree &T, const uint32_t (&ref)[NL], const uint32_t (&cnt)[NL], int lane,
                                            const pc_seg_dev &S, const pc_knn_dev &K, pc_seg_geo &G, pc_knn_wlist &W)
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
            e = pc_seg_exact_d2(p[j].x, p[j].y, p[j].z, G);
            id = (uint32_t)__float_as_int(p[j].w);
            have = e <= S.r2;
        }
        const float before = W.thr;
        pc_knn_warp_insert(have, e, id, lane, K, W);
        if (W.thr != before) pc_seg_set_thr(W.thr, G);
    }
}

// the frontier walk of pc_knn_warp_search with the segment's node test
__device__ __forceinline__ void pc_seg_search(const pc_tree &T, const pc_seg_dev &S, const pc_knn_dev &K, uint2 *__restrict__ F,
                                              int lane, pc_seg_geo &G, pc_knn_wlist &W)
{
    const uint32_t lt = (1u << lane) - 1u;
    const int n_seed = (int)T.seeds[0], n_seed_leaf = (int)T.seeds[1];
    for (int base = 0; base < n_seed_leaf; base += 32) {
        uint32_t ref[1] = { 0u }, cnt[1] = { 0u };
        if (base + lane < n_seed_leaf) { ref[0] = T.seeds[PC_SEED_LEAF + 2 * (base + lane)]; cnt[0] = T.seeds[PC_SEED_LEAF + 2 * (base + lane) + 1]; }
        pc_seg_scan<1>(T, ref, cnt, lane, S, K, G, W);
    }
    if (lane < n_seed) F[lane] = make_uint2(T.seeds[PC_SEED_INNER + lane], 0u);
    int size = n_seed;
    __syncwarp();
    while (size > 0) {
        const int take = (size + 32 + PC_STACK <= PC_KNN_FRONT) ? min(size, 32) : 1;
        bool active = lane < take;
        uint2 en = make_uint2(0u, 0u);
        if (active) en = F[size - 1 - lane];
        size -= take;
        __syncwarp();
        active = active && __uint_as_float(en.y) <= G.thr2;
        float dn = INFINITY, df = INFINITY;
        uint32_t cn = 0, cf = 0;
        uint32_t ref[2] = { 0u, 0u }, cnt[2] = { 0u, 0u };
        if (active) {
            const pc_rec rec = pc_load_rec(T.rec + 4ull * en.x);
            const float d0 = pc_seg_box(rec.L[0], rec.L[2], rec.L[4], rec.H[0], rec.H[2], rec.H[4], G);
            const float d1 = pc_seg_box(rec.L[1], rec.L[3], rec.L[5], rec.H[1], rec.H[3], rec.H[5], G);
            const bool first0 = d0 <= d1;
            const uint32_t r0 = pc_rec_ref(rec, 0), r1 = pc_rec_ref(rec, 1);
            const uint32_t rn = first0 ? r0 : r1, rf = first0 ? r1 : r0;
            const uint32_t kn = pc_rec_cnt(rec, first0 ? 0 : 1), kf = pc_rec_cnt(rec, first0 ? 1 : 0);
            const float dnn = fminf(d0, d1), dff = fmaxf(d0, d1);
            if (dnn <= G.thr2) {
                if (rn & PC_REF_LEAF) { ref[0] = rn; cnt[0] = kn; }
                else { cn = rn; dn = dnn; }
            }
            if (dff <= G.thr2) {
                if (rf & PC_REF_LEAF) { ref[1] = rf; cnt[1] = kf; }
                else { cf = rf; df = dff; }
            }
        }
        if (__ballot_sync(PC_FULL_MASK, (cnt[0] | cnt[1]) != 0u)) pc_seg_scan<2>(T, ref, cnt, lane, S, K, G, W);
        const bool wn = dn <= G.thr2, wf = df <= G.thr2;
        const uint32_t mf = __ballot_sync(PC_FULL_MASK, wf), mn = __ballot_sync(PC_FULL_MASK, wn);
        const int nf = __popc(mf), nn = __popc(mn);
        if (wf) F[size + __popc(mf & lt)] = make_uint2(cf, __float_as_uint(df));
        if (wn) F[size + nf + (nn - 1 - __popc(mn & lt))] = make_uint2(cn, __float_as_uint(dn));
        size += nf + nn;
        __syncwarp();
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
    pc_knn_dev K;
    K.k = 1; K.r2 = S.r2; K.bound_thr = S.bound_thr; K.packet_split = 0.f; K.defer_count = nullptr; K.defer_list = nullptr;
    const long long m_search = m_eff ? (long long)*m_eff : (long long)m;
    const long long n_warps = (long long)gridDim.x * PC_SEG_WARPS;
    for (long long t = (long long)blockIdx.x * PC_SEG_WARPS + w; t < m_search; t += n_warps) {
        const uint32_t slot = ordered ? __float_as_uint(ordered[t].w) : perm ? perm[t] : (uint32_t)t;
        const float *a = a_xyz + (size_t)slot * stride, *b = b_xyz + (size_t)slot * stride;
        const float av[3] = { a[0], a[1], a[2] }, bv[3] = { b[0], b[1], b[2] };
        const bool finite = isfinite(av[0]) && isfinite(av[1]) && isfinite(av[2]) && isfinite(bv[0]) && isfinite(bv[1]) && isfinite(bv[2]);
        pc_knn_wlist W;
        W.ld = W.kd = INFINITY; W.li = W.ki = PC_KNN_NONE; W.thr = S.bound_thr;
        if (finite && T.n_points > 0) {
            pc_seg_geo G;
            pc_seg_setup(av, bv, G);
            pc_seg_set_thr(W.thr, G);
            pc_seg_search(T, S, K, s_front[w], lane, G, W);
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
