// query_kernels.cuh -- exact nearest / radius queries over the prefix-split tree (build_kernels.cuh).
//
// Replaces kd_nearest_i / kd_nearest3 (Utils/kdtree/src/kdtree.c:345-457,493-500) and the epilogue of
// safeRegionRrtStar::radiusSearch (Planner/src/corridor_finder.cpp:113-133).
//
// Exactness: boxes and points are filtered in fp32 against `thr`, an upper bound of the current best fp64
// distance inflated by 2^-20 (fp32 evaluation error of d2 is < 2^-22 relative, so no candidate whose fp64
// distance is <= best can be filtered out); survivors are re-evaluated in fp64 with un-fused
// __dsub_rn/__dmul_rn/__dadd_rn in the reference's operation order and ranked by (d2, original index).
//
// Three walks, all returning identical results:
//   pc_nearest_traverse     one thread per query, near-first descent with a per-thread stack (unordered large batches)
//   pc_packet_traverse<NQ>  one WARP walks the tree once for 32 * NQ neighbouring queries of a curve-ordered batch
//   pc_query_coop_kernel    a GROUP of 8 / 16 / 32 lanes per query (small batches, the planner's one-query calls)
#pragma once
#include "common.cuh"
#include "build_kernels.cuh"
#include "radix_sort.cuh"

#ifndef PC_QUERY_THREADS
#define PC_QUERY_THREADS 128
#endif
#define PC_STACK 96                            // tree depth <= key bits (<= 63) + position bits of coincident points (<= 31)
#define PC_THR_SLACK 1.00000095367431640625f   // 1 + 2^-20
#define PC_NO_NODE 0xffffffffu
#ifndef PC_PACKET_MIN_CTAS
#define PC_PACKET_MIN_CTAS 10       // resident CTAs per SM the packet kernels are compiled for (<= 48 registers).  With the packed
                                    // arithmetic the kernel waits on record loads more than on issue slots: 10 CTAs 0.77 ms,
                                    // 9: 0.80, 8: 0.82, 12 (40 registers, the hot loop spills): 1.03 (profiles/r2_variants_ab.txt)
#endif
#ifndef PC_PACKET_PREFETCH
#define PC_PACKET_PREFETCH 0        // 1: when a record arrives, pull the records of its two children towards L1 (measured:
                                    // +10 % search time -- the extra requests cost more than the latency they hide)
#endif

struct pc_tree {
    const float4 *__restrict__ rec;      // inner node i -> rec[4i .. 4i+3] = [min0 | max0 | min1 | max1], children in the .w words
    const float4 *__restrict__ points;   // curve order, (x, y, z, original index); PC_LEAF pad copies of the last point behind
    int64_t n_points;
    uint32_t root;                       // child reference of the whole cloud: inner node 0, or the leaf PC_REF_LEAF | 0
    uint32_t root_count;                 // number of points when the root is a leaf
    const uint32_t *__restrict__ seeds;  // top of the tree expanded to <= 32 inner nodes (+ leaves met on the way): pc_tree_seed_kernel
};

// ---- packed fp32x2 arithmetic (Blackwell: FADD2 / FFMA2) ------------------------------------------------------------------
// sm_100 adds packed add.f32x2 / fma.f32x2 (SASS FADD2 / FFMA2): two independent IEEE fp32 operations per instruction on a
// register pair, and an operand may be a scalar that the instruction broadcasts to both halves.  The records interleave the
// two children per axis (build_kernels.cuh), so the distance of one query to BOTH child boxes takes 15 instructions instead
// of 24 -- in every walk, whatever the number of queries per lane -- and the 64-query packets also scan a leaf for their two
// queries at once.  Each half is an ordinary fp32 operation: the results are bit-identical with scalar code.
__device__ __forceinline__ float2 pc_add2(float2 a, float2 b)
{
    float2 r;
    asm("{ .reg .b64 ra, rb, rc; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; add.rn.f32x2 rc, ra, rb; mov.b64 {%0, %1}, rc; }"
        : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return r;
}
__device__ __forceinline__ float2 pc_fma2(float2 a, float2 b, float2 c)
{
    float2 r;
    asm("{ .reg .b64 ra, rb, rc, rd; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; mov.b64 rc, {%6, %7}; fma.rn.f32x2 rd, ra, rb, rc; mov.b64 {%0, %1}, rd; }"
        : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return r;
}

// one record: two 256-bit read-only loads (sm_100: LDG.E.256).  L = [min0.x min1.x min0.y min1.y min0.z min1.z ref0 ref1],
// H = [max0.x max1.x max0.y max1.y max0.z max1.z cnt0 cnt1]
struct pc_rec { float L[8], H[8]; };
__device__ __forceinline__ pc_rec pc_load_rec(const float4 *__restrict__ rec)
{
    pc_rec r;
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(r.L[0]), "=f"(r.L[1]), "=f"(r.L[2]), "=f"(r.L[3]), "=f"(r.L[4]), "=f"(r.L[5]), "=f"(r.L[6]), "=f"(r.L[7]) : "l"(rec));
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(r.H[0]), "=f"(r.H[1]), "=f"(r.H[2]), "=f"(r.H[3]), "=f"(r.H[4]), "=f"(r.H[5]), "=f"(r.H[6]), "=f"(r.H[7]) : "l"(rec + 2));
    return r;
}
__device__ __forceinline__ uint32_t pc_rec_ref(const pc_rec &r, int c) { return __float_as_uint(r.L[6 + c]); }
__device__ __forceinline__ uint32_t pc_rec_cnt(const pc_rec &r, int c) { return __float_as_uint(r.H[6 + c]); }

// squared distances of one query to the two child boxes of a record: (.x = child 0, .y = child 1).  Per axis
// max(min - q, q - max, 0), then dz^2 + (dy^2 + dx^2) with fused multiply-adds, as the scalar formula did.
__device__ __forceinline__ float2 pc_rec_d2(const pc_rec &r, float qx, float qy, float qz)
{
    const float2 m1 = make_float2(-1.f, -1.f), zero = make_float2(0.f, 0.f);
    float2 t1 = pc_add2(make_float2(r.L[0], r.L[1]), make_float2(-qx, -qx)), t2 = pc_fma2(make_float2(r.H[0], r.H[1]), m1, make_float2(qx, qx));
    const float2 dx = make_float2(fmaxf(fmaxf(t1.x, t2.x), 0.0f), fmaxf(fmaxf(t1.y, t2.y), 0.0f));
    t1 = pc_add2(make_float2(r.L[2], r.L[3]), make_float2(-qy, -qy)); t2 = pc_fma2(make_float2(r.H[2], r.H[3]), m1, make_float2(qy, qy));
    const float2 dy = make_float2(fmaxf(fmaxf(t1.x, t2.x), 0.0f), fmaxf(fmaxf(t1.y, t2.y), 0.0f));
    t1 = pc_add2(make_float2(r.L[4], r.L[5]), make_float2(-qz, -qz)); t2 = pc_fma2(make_float2(r.H[4], r.H[5]), m1, make_float2(qz, qz));
    const float2 dz = make_float2(fmaxf(fmaxf(t1.x, t2.x), 0.0f), fmaxf(fmaxf(t1.y, t2.y), 0.0f));
    return pc_fma2(dz, dz, pc_fma2(dy, dy, pc_fma2(dx, dx, zero)));
}

// the reference's fp64 expression: s = 0; s += (px-qx)^2; s += (py-qy)^2; s += (pz-qz)^2  (kdtree.c:379-382)
__device__ __forceinline__ double pc_exact_d2(float px, float py, float pz, double qx, double qy, double qz)
{
    double dx = __dsub_rn((double)px, qx), dy = __dsub_rn((double)py, qy), dz = __dsub_rn((double)pz, qz);
    double s = __dmul_rn(dx, dx);
    s = __dadd_rn(s, __dmul_rn(dy, dy));
    s = __dadd_rn(s, __dmul_rn(dz, dz));
    return s;
}

__device__ __forceinline__ float pc_thr_from(double best)
{
    return __fmul_ru(__double2float_ru(best), PC_THR_SLACK);
}

struct pc_best {
    double d2;     // +inf until a point is accepted
    int32_t idx;   // -1 until a point is accepted
    float thr;     // fp32 filter threshold (inclusive); < 0: this lane has no query
};

__device__ __forceinline__ void pc_consider(const float4 p, float d, float qx, float qy, float qz, pc_best &b)
{
    if (d <= b.thr) {
        const double e = pc_exact_d2(p.x, p.y, p.z, (double)qx, (double)qy, (double)qz);
        const int32_t id = __float_as_int(p.w);
        if (e < b.d2 || (e == b.d2 && (uint32_t)id < (uint32_t)b.idx)) {
            b.d2 = e; b.idx = id; b.thr = fminf(b.thr, pc_thr_from(e));
        }
    }
}

// fp64 re-check of a scanned leaf for one query.  A point can be the exact minimiser only if its fp32 d2 is within the
// fp32 error of the leaf's fp32 minimum dmin: any point with d2 > dmin (1 + 2^-20) + 2^-147 (relative error < 2^-22, and
// the absolute 2^-147 covers fp32 underflow of tiny distances) has a larger fp64 distance than the minimum's point.  So
// only the points inside that margin (and inside thr) -- almost always one -- are re-evaluated, in a loop with ONE fp64
// site instead of one per point; the point is read again (an L1 hit) rather than held in registers.  The result is the
// one every point's re-check would give: smallest (d2, original index).
__device__ __forceinline__ void pc_exact_leaf(const float4 *__restrict__ pts, const float (&d)[PC_LEAF], float dmin,
                                              float qx, float qy, float qz, pc_best &b)
{
    if (!(dmin <= b.thr)) return;          // one branch for the whole leaf: after the first leaves almost never taken
    const float cut = fminf(b.thr, __fmaf_ru(dmin, PC_THR_SLACK, 4.0f * FLT_TRUE_MIN));
    uint32_t cand = 0;
#pragma unroll
    for (int i = 0; i < PC_LEAF; i++) cand |= (d[i] <= cut ? 1u : 0u) << i;
    const double dqx = qx, dqy = qy, dqz = qz;
    while (cand) {
        const float4 p = __ldg(pts + (__ffs(cand) - 1));
        cand &= cand - 1u;
        const double e = pc_exact_d2(p.x, p.y, p.z, dqx, dqy, dqz);
        const int32_t id = __float_as_int(p.w);
        if (e < b.d2 || (e == b.d2 && (uint32_t)id < (uint32_t)b.idx)) { b.d2 = e; b.idx = id; }
    }
    b.thr = fminf(b.thr, pc_thr_from(b.d2));
}

// Leaf scan for NQ queries of one lane: PC_LEAF consecutive points from an arbitrary start (128-bit loads).  The points
// behind the leaf's own count are real points of the cloud too (or pad copies of the last one), so scanning them cannot
// break exactness.
template <int NQ>
__device__ __forceinline__ void pc_scan_leaf(const float4 *__restrict__ pts, const float (&q)[NQ][3], pc_best (&b)[NQ])
{
    float4 p[PC_LEAF];
    float d[NQ][PC_LEAF], dmin[NQ];
#pragma unroll
    for (int i = 0; i < PC_LEAF; i++) p[i] = __ldg(pts + i);
#pragma unroll
    for (int j = 0; j < NQ; j++) {
        dmin[j] = FLT_MAX;
#pragma unroll
        for (int i = 0; i < PC_LEAF; i++) {
            const float dx = p[i].x - q[j][0], dy = p[i].y - q[j][1], dz = p[i].z - q[j][2];
            d[j][i] = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
            dmin[j] = fminf(dmin[j], d[j][i]);
        }
    }
#pragma unroll
    for (int j = 0; j < NQ; j++) pc_exact_leaf(pts, d[j], dmin[j], q[j][0], q[j][1], q[j][2], b[j]);
}

// the same leaf scan for the two queries of a lane, distances two at a time (nq* = (-qa, -qb) per axis)
__device__ __forceinline__ void pc_scan_leaf_x2(const float4 *__restrict__ pts, float2 nqx, float2 nqy, float2 nqz, pc_best (&b)[2])
{
    float da[PC_LEAF], db[PC_LEAF];
    const float2 zero = make_float2(0.f, 0.f);
    float mina = FLT_MAX, minb = FLT_MAX;
#pragma unroll
    for (int i = 0; i < PC_LEAF; i++) {
        const float4 p = __ldg(pts + i);
        const float2 ex = pc_add2(make_float2(p.x, p.x), nqx), ey = pc_add2(make_float2(p.y, p.y), nqy),
                     ez = pc_add2(make_float2(p.z, p.z), nqz);
        const float2 dd = pc_fma2(ez, ez, pc_fma2(ey, ey, pc_fma2(ex, ex, zero)));
        da[i] = dd.x; db[i] = dd.y;
        mina = fminf(mina, dd.x); minb = fminf(minb, dd.y);
    }
    pc_exact_leaf(pts, da, mina, -nqx.x, -nqy.x, -nqz.x, b[0]);
    pc_exact_leaf(pts, db, minb, -nqx.y, -nqy.y, -nqz.y, b[1]);
}

// Core traversal of one query by one thread.  On entry b holds the initial bound (d2 = +inf, idx = -1, thr = bound).
__device__ __forceinline__ void pc_nearest_traverse(const pc_tree &T, float qx, float qy, float qz, pc_best &b)
{
    const float qv[1][3] = { { qx, qy, qz } };
    pc_best bb[1] = { b };
    if (T.root & PC_REF_LEAF) { pc_scan_leaf<1>(T.points + (T.root & ~PC_REF_LEAF), qv, bb); b = bb[0]; return; }
    uint32_t stack_ref[PC_STACK];
    float stack_d[PC_STACK];
    int sp = 0;
    uint32_t ref = T.root;
    for (;;) {
        const pc_rec rec = pc_load_rec(T.rec + 4ull * ref);
        const float2 dd = pc_rec_d2(rec, qx, qy, qz);
        const float d0 = dd.x, d1 = dd.y;
        const uint32_t r0 = pc_rec_ref(rec, 0), r1 = pc_rec_ref(rec, 1);
        const bool first0 = d0 <= d1;
        const uint32_t rn = first0 ? r0 : r1, rf = first0 ? r1 : r0;
        const float dn = fminf(d0, d1), df = fmaxf(d0, d1);
        ref = PC_NO_NODE;
        if (dn <= bb[0].thr) {
            if (rn & PC_REF_LEAF) pc_scan_leaf<1>(T.points + (rn & ~PC_REF_LEAF), qv, bb);
            else ref = rn;
        }
        if (df <= bb[0].thr) {
            if (rf & PC_REF_LEAF) pc_scan_leaf<1>(T.points + (rf & ~PC_REF_LEAF), qv, bb);
            else if (ref == PC_NO_NODE) ref = rf;
            else { stack_ref[sp] = rf; stack_d[sp] = df; sp++; }
        }
        if (ref != PC_NO_NODE) continue;
        // pop until a still-promising node is found
        while (sp > 0) {
            sp--;
            if (stack_d[sp] <= bb[0].thr) { ref = stack_ref[sp]; break; }
        }
        if (ref == PC_NO_NODE) break;
    }
    b = bb[0];
}

// ---- radiusSearch pieces ------------------------------------------------------------------------------
struct pc_radius_dev {
    double search_margin, max_radius, sample_range;
    double sx, sy, sz;
    float bound_thr;    // fp32 threshold on d2 for the bounded search (FLT_MAX when unbounded)
    int bounded;        // PC_RADIUS_BOUNDED: out_idx = -1 wherever the radius clamps to max_radius
    int pcl_float;      // PC_ARITH_PCL_FLOAT: d2 rounded to float32 and float32 sqrt, as PCL's interface makes the reference compute
    double range_lo2, range_hi2;   // (sample_range + max_radius)^2 * (1 -+ 1e-12): outside this band the early-out needs no sqrt
    float packet_split;            // unbounded packet walks: largest Chebyshev distance inside one shared walk (0 = no limit); packets
    unsigned long long *defer_count;   // beyond it are queued here by pc_query_packet_kernel<PC_KIND_NEAREST> for
    uint32_t *defer_list;              // pc_query_deferred_kernel
};

// radiusSearch epilogue on a finished search (corridor_finder.cpp:131-132); nothing found inside the bound => clamp
__device__ __forceinline__ double pc_radius_epilogue(const pc_best &b, const pc_radius_dev &R)
{
    if (b.idx < 0) return R.max_radius;
    // corridor_finder.cpp:131: sqrt(pointRadiusSquaredDistance[0]) - search_margin.  The reference's distance arrives in a
    // std::vector<float> and `sqrt` resolves to the float overload; PC_ARITH_PCL_FLOAT reproduces exactly that, the default
    // keeps the kd-tree's double precision (the north star's parity target, 1e-6 relative of the float variant).
    double radius = R.pcl_float ? __dsub_rn((double)__fsqrt_rn(__double2float_rn(b.d2)), R.search_margin)
                                : __dsub_rn(__dsqrt_rn(b.d2), R.search_margin);
    return radius < R.max_radius ? radius : R.max_radius;
}

// radiusSearch early-out (corridor_finder.cpp:115-116): |p - start| > sample_range + max_radius
__device__ __forceinline__ bool pc_radius_early_out(double px, double py, double pz, const pc_radius_dev &R)
{
    if (R.sample_range < 0.0) return false;
    double dx = __dsub_rn(px, R.sx), dy = __dsub_rn(py, R.sy), dz = __dsub_rn(pz, R.sz);
    double s = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    // sqrt is monotone and correctly rounded (relative error < 2^-53), so away from the boundary the comparison of the
    // squares decides; only a point within 1e-12 (relative) of the sensing sphere takes the reference's own expression
    if (s > R.range_hi2) return true;
    if (s < R.range_lo2) return false;
    return __dsqrt_rn(s) > __dadd_rn(R.sample_range, R.max_radius);
}

#define PC_KIND_NEAREST 0
#define PC_KIND_RADIUS 1

// result of a query that needs no search: empty cloud (kd_nearest3 -> NULL; corridor_finder.cpp:118-120) or outside the
// sensing range (corridor_finder.cpp:115-116)
template <int KIND>
__device__ __forceinline__ void pc_write_trivial(const pc_radius_dev &R, uint32_t k, int32_t *out_idx, float *out_f)
{
    if (out_idx) out_idx[k] = -1;
    if (out_f) out_f[k] = (KIND == PC_KIND_RADIUS) ? (float)__dsub_rn(R.max_radius, R.search_margin) : INFINITY;
}

template <int KIND>
__device__ __forceinline__ void pc_write_result(const pc_radius_dev &R, const pc_best &b, uint32_t k, int32_t *out_idx, float *out_f)
{
    if (KIND == PC_KIND_RADIUS) {
        const double radius = pc_radius_epilogue(b, R);
        if (out_f) out_f[k] = (float)radius;
        if (out_idx) out_idx[k] = (R.bounded && !(radius < R.max_radius)) ? -1 : b.idx;
    } else {
        if (out_idx) out_idx[k] = b.idx;
        if (out_f) out_f[k] = (float)b.d2;
    }
}

// ---- one thread per query -------------------------------------------------------------------------------------------
// perm (nullable): process query perm[t] in slot t (curve-ordered batches); results go to the original slot.
// ordered (nullable, instead of perm): slot t holds the query itself, (x, y, z, original slot) -- the cell-binned batch.
// m_eff (nullable): device-side number of leading entries of perm that need a search (the rest were answered by the
// ordering pass).
template <int KIND>
__global__ void __launch_bounds__(PC_QUERY_THREADS)
pc_query_simple_kernel(pc_tree T, pc_radius_dev R, const float *__restrict__ q, int64_t m, int qstride,
                       const uint32_t *__restrict__ perm, const float4 *__restrict__ ordered, const unsigned long long *__restrict__ m_eff,
                       int32_t *__restrict__ out_idx, float *__restrict__ out_f)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m || (m_eff && t >= (int64_t)*m_eff)) return;
    uint32_t k;
    float qx, qy, qz;
    if (ordered) { const float4 v = __ldg(ordered + t); qx = v.x; qy = v.y; qz = v.z; k = __float_as_uint(v.w); }
    else { k = perm ? perm[t] : (uint32_t)t; const float *qq = q + (size_t)k * qstride; qx = qq[0]; qy = qq[1]; qz = qq[2]; }
    bool search = T.n_points > 0;
    if (KIND == PC_KIND_RADIUS && search && !m_eff && pc_radius_early_out((double)qx, (double)qy, (double)qz, R)) search = false;
    if (!search) { pc_write_trivial<KIND>(R, k, out_idx, out_f); return; }
    pc_best b; b.d2 = INFINITY; b.idx = -1; b.thr = (KIND == PC_KIND_RADIUS) ? R.bound_thr : FLT_MAX;
    pc_nearest_traverse(T, qx, qy, qz, b);
    pc_write_result<KIND>(R, b, k, out_idx, out_f);
}

// ---- warp packets ---------------------------------------------------------------------------------------------------
// After the ordering pass the 32 * NQ queries of a warp lie in one small cell of the curve, so their searches visit almost
// the same nodes.  The warp therefore walks the tree ONCE for all of them: one stack of postponed children for the whole warp
// (local memory at a warp-uniform index, see below), every node record loaded once at a warp-uniform address, each lane
// testing its own NQ queries against it; a child is entered when ANY query still needs it (ballot), the nearer child is
// chosen by a majority vote of the lanes' first queries.  Control flow is warp-uniform, so all 32 lanes are active at every
// step; the price is that a lane also visits nodes only its neighbours needed.
// NQ = 2 halves the record bytes and the control instructions per query-visit (dense batches); NQ = 1 keeps packets small
// for sparser batches.  A child that is a leaf is scanned on the spot; only inner nodes are pushed.
// Measured and dropped in round 1 (profiles/r1_sweep3/4/6/8*): rejecting stale stack entries with per-entry minimum
// distances, a 32-wide sideways test of descendants against the packet's box, a 4-ary walk, letting both queries of a lane
// vote, packed __reduce_add_sync votes, most-wanted-child-first ordering, far-child prefetch on push.
// Must be called by all 32 lanes of a warp, converged; lanes without a query pass thr < 0 and take part in the votes only.
template <int NQ>
__device__ __forceinline__ void pc_packet_traverse(const pc_tree &T, const float (&q)[NQ][3], pc_best (&b)[NQ], int lane)
{
    bool any = false;
#pragma unroll
    for (int j = 0; j < NQ; j++) any = any || b[j].thr >= 0.f;
    if (__ballot_sync(PC_FULL_MASK, any) == 0) return;
    if (T.root & PC_REF_LEAF) { pc_scan_leaf<NQ>(T.points + (T.root & ~PC_REF_LEAF), q, b); return; }
    // NQ == 2: the lane's two queries packed per axis, negated, for the leaf scans (pc_scan_leaf_x2)
    const float2 nqx = make_float2(-q[0][0], -q[NQ - 1][0]), nqy = make_float2(-q[0][1], -q[NQ - 1][1]), nqz = make_float2(-q[0][2], -q[NQ - 1][2]);
    auto scan = [&](const float4 *pts) {
        if constexpr (NQ == 2) pc_scan_leaf_x2(pts, nqx, nqy, nqz, b);
        else pc_scan_leaf<NQ>(pts, q, b);
    };
    // The warp's stack of postponed children lives in LOCAL memory, the same copy in every lane at a warp-uniform index: one
    // coalesced 128-byte STL per push, one LDL per pop (L1-resident), no registers, no shuffles.  Measured against three
    // registers per lane read back with __shfl_sync (which ptxas spilled at 48 registers anyway): 0.81 -> 0.77 ms; against
    // shared memory: 0.93 ms (profiles/r2_variants_ab.txt).
    uint32_t stack[PC_STACK];
    int sp = 0;
    uint32_t ref = T.root;
    for (;;) {
        const pc_rec rec = pc_load_rec(T.rec + 4ull * ref);
#if PC_PACKET_PREFETCH
        {   // the next visit is one of the two children (or a stack entry): start their records' trip from L2 now, while the
            // box tests and votes below run (a leaf reference fetches a line of the points instead, also the next access)
            const uint32_t c0 = pc_rec_ref(rec, 0), c1 = pc_rec_ref(rec, 1);
            const float4 *a0 = (c0 & PC_REF_LEAF) ? T.points + (c0 & ~PC_REF_LEAF) : T.rec + 4ull * c0;
            const float4 *a1 = (c1 & PC_REF_LEAF) ? T.points + (c1 & ~PC_REF_LEAF) : T.rec + 4ull * c1;
            asm volatile("prefetch.global.L1 [%0];" ::"l"(a0));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(a1));
        }
#endif
        float d0[NQ], d1[NQ];
        bool want0 = false, want1 = false;
        if constexpr (NQ == 2) {
            // from the packed negated copies, so that the queries are held once (registers: the kernel runs 10 CTAs per SM)
            const float2 da = pc_rec_d2(rec, -nqx.x, -nqy.x, -nqz.x), db = pc_rec_d2(rec, -nqx.y, -nqy.y, -nqz.y);
            d0[0] = da.x; d1[0] = da.y; d0[1] = db.x; d1[1] = db.y;
        } else {
#pragma unroll
            for (int j = 0; j < NQ; j++) {
                const float2 dd = pc_rec_d2(rec, q[j][0], q[j][1], q[j][2]);       // both children at once
                d0[j] = dd.x; d1[j] = dd.y;
            }
        }
#pragma unroll
        for (int j = 0; j < NQ; j++) {
            want0 = want0 || d0[j] <= b[j].thr;
            want1 = want1 || d1[j] <= b[j].thr;
        }
        const uint32_t w0 = __ballot_sync(PC_FULL_MASK, want0);
        const uint32_t w1 = __ballot_sync(PC_FULL_MASK, want1);
        uint32_t next = PC_NO_NODE;
        if (w0 | w1) {
            const bool both = w0 != 0 && w1 != 0;
            bool first0 = w1 == 0;
            if (both) {
                // majority vote of the interested lanes' FIRST queries (not needed when only one child is wanted)
                const uint32_t ia = __ballot_sync(PC_FULL_MASK, d0[0] <= b[0].thr || d1[0] <= b[0].thr);
                const uint32_t pa = __ballot_sync(PC_FULL_MASK, d0[0] <= d1[0]) & ia;
                first0 = 2 * __popc(pa) >= __popc(ia);
            }
            const uint32_t r0 = pc_rec_ref(rec, 0), r1 = pc_rec_ref(rec, 1);
            const uint32_t rn = first0 ? r0 : r1, rf = first0 ? r1 : r0;
            if (rn & PC_REF_LEAF) scan(T.points + (rn & ~PC_REF_LEAF));
            else next = rn;
            if (both) {
                if (rf & PC_REF_LEAF) {
                    bool again = false;          // the near leaf may have tightened the bounds
#pragma unroll
                    for (int j = 0; j < NQ; j++) again = again || (first0 ? d1[j] : d0[j]) <= b[j].thr;
                    if (__ballot_sync(PC_FULL_MASK, again)) scan(T.points + (rf & ~PC_REF_LEAF));
                } else if (next != PC_NO_NODE) {
                    stack[sp] = rf;
                    sp++;
                } else next = rf;
            }
        }
        if (next != PC_NO_NODE) { ref = next; continue; }
        if (sp == 0) break;
        sp--;
        ref = stack[sp];
    }
}

template <int KIND, int NQ>
__global__ void __launch_bounds__(PC_QUERY_THREADS, NQ <= 2 ? PC_PACKET_MIN_CTAS : PC_PACKET_MIN_CTAS / 2)
pc_query_packet_kernel(pc_tree T, pc_radius_dev R, const float *__restrict__ q, int64_t m, int qstride,
                       const uint32_t *__restrict__ perm, const float4 *__restrict__ ordered, const unsigned long long *__restrict__ m_eff,
                       int32_t *__restrict__ out_idx, float *__restrict__ out_f)
{
    const int lane = threadIdx.x & 31;
    const long long m_search = m_eff ? (long long)*m_eff : (long long)m;
    const long long warp_id = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long base = warp_id * (32 * NQ);
    if (base >= m_search) return;                           // whole warp past the end
    float qv[NQ][3];
    uint32_t k[NQ];
    bool valid[NQ];
    pc_best b[NQ];
#pragma unroll
    for (int j = 0; j < NQ; j++) {
        const long long t = base + 32 * j + lane;
        valid[j] = t < m_search;
        k[j] = 0u; qv[j][0] = qv[j][1] = qv[j][2] = 0.f;
        b[j].d2 = INFINITY; b[j].idx = -1; b[j].thr = -1.0f;      // thr < 0: this slot needs nothing
        if (valid[j]) {
            if (ordered) {
                const float4 v = __ldcs(ordered + t);          // coalesced: the batch was gathered into cell order; read once
                qv[j][0] = v.x; qv[j][1] = v.y; qv[j][2] = v.z; k[j] = __float_as_uint(v.w);
            } else {
                k[j] = perm ? perm[t] : (uint32_t)t;
                const float *qq = q + (size_t)k[j] * qstride;
                qv[j][0] = qq[0]; qv[j][1] = qq[1]; qv[j][2] = qq[2];
            }
            bool search = T.n_points > 0;
            if (KIND == PC_KIND_RADIUS && search && !m_eff && pc_radius_early_out((double)qv[j][0], (double)qv[j][1], (double)qv[j][2], R)) search = false;
            if (search) b[j].thr = (KIND == PC_KIND_RADIUS) ? R.bound_thr : FLT_MAX;
            else { pc_write_trivial<KIND>(R, k[j], out_idx, out_f); valid[j] = false; }
        }
    }
    if ((KIND == PC_KIND_NEAREST || !R.bounded) && R.packet_split > 0.f) {
        // An UNBOUNDED walk is shared well only by queries that lie close together: a lane far from the others keeps an
        // infinite (then very loose) bound until the walk -- steered by the majority -- happens to come near it, and until then
        // it wants every node.  Packets are cut from the curve order at fixed positions, so a few straddle a jump of the curve
        // (the 3-D Hilbert order of a flat map leaves and re-enters the slab of the map) or, in pc_batch_shard mode, two cells of
        // the rank's share that are not neighbours; one such packet can walk a large part of the tree, alone, for milliseconds
        // (C5 split over 8 ranks: half of the ranks took 12 ms instead of 6).  A packet with a query farther than packet_split
        // (Chebyshev; some packet extents at the batch's density) from its first one is not walked here: it is queued for
        // pc_query_deferred_kernel, where every query walks alone.
        const float ax = __shfl_sync(PC_FULL_MASK, qv[0][0], 0), ay = __shfl_sync(PC_FULL_MASK, qv[0][1], 0), az = __shfl_sync(PC_FULL_MASK, qv[0][2], 0);
        bool far = false;
#pragma unroll
        for (int j = 0; j < NQ; j++)
            far = far || (b[j].thr >= 0.f && fmaxf(fmaxf(fabsf(qv[j][0] - ax), fabsf(qv[j][1] - ay)), fabsf(qv[j][2] - az)) > R.packet_split);
        if (__any_sync(PC_FULL_MASK, far)) {
            if (lane == 0) R.defer_list[atomicAdd(R.defer_count, 1ull)] = (uint32_t)warp_id;
            return;
        }
    }
    pc_packet_traverse<NQ>(T, qv, b, lane);
#pragma unroll
    for (int j = 0; j < NQ; j++)
        if (valid[j]) pc_write_result<KIND>(R, b[j], k[j], out_idx, out_f);
}

// The packets pc_query_packet_kernel<PC_KIND_NEAREST, NQ> put aside (R.defer_list / R.defer_count; `per_packet` = 32 NQ queries
// each): every query walks the tree on its own, one thread per query (pc_nearest_traverse, the walk of
// pc_query_simple_kernel) -- robust whatever the shape of the packet, and the few thousand walks of a typical call run side
// by side.  (Measured alternative: walking such a packet in groups of nearby queries -- a group that is still spread out is
// as slow as the packet was, and at a tight grouping distance thousands of packets queue for a handful of warps.)
#define PC_DEFER_CTAS_PER_SM 4

template <int KIND>
__global__ void __launch_bounds__(PC_QUERY_THREADS)
pc_query_deferred_kernel(pc_tree T, pc_radius_dev R, const float *__restrict__ q, int64_t m, int qstride, int per_packet,
                         const uint32_t *__restrict__ perm, const float4 *__restrict__ ordered, const unsigned long long *__restrict__ m_eff,
                         int32_t *__restrict__ out_idx, float *__restrict__ out_f)
{
    const long long m_search = m_eff ? (long long)*m_eff : (long long)m;
    const unsigned long long total = *R.defer_count * (unsigned long long)per_packet;
    const unsigned long long n_threads = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long e = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += n_threads) {
        const long long t = (long long)R.defer_list[e / (unsigned)per_packet] * per_packet + (long long)(e % (unsigned)per_packet);
        if (t >= m_search) continue;
        uint32_t k;
        float qx, qy, qz;
        if (ordered) { const float4 v = ordered[t]; qx = v.x; qy = v.y; qz = v.z; k = __float_as_uint(v.w); }
        else { k = perm ? perm[t] : (uint32_t)t; const float *qq = q + (size_t)k * qstride; qx = qq[0]; qy = qq[1]; qz = qq[2]; }
        pc_best b; b.d2 = INFINITY; b.idx = -1; b.thr = FLT_MAX;
        pc_nearest_traverse(T, qx, qy, qz, b);
        pc_write_result<KIND>(R, b, k, out_idx, out_f);
    }
}

// ---- a GROUP of lanes per query (small batches) -----------------------------------------------------------------------
// The planner's own loop asks for ONE radius per call (corridor_finder.cpp:404), and then a search is a chain of dependent
// loads: tens of node visits of ~0.5 us each with one thread per query.  Here G lanes (a whole warp for the smallest batches,
// 16 or 8 lanes when there are more queries than the GPU holds warps) work on the same query: the open inner nodes sit on a
// LIFO frontier in shared memory, every step the group takes the (up to) G most recently pushed -- deepest, nearest -- nodes,
// one per lane, tests their two child boxes, scans the children that are leaves, shares the tightened bound with one warp
// reduction and pushes the surviving inner children, the nearer ones on top.  The number of dependent steps drops from the
// number of visits to roughly the depth of the tree.
// Exactness as everywhere: fp32 filter against the shared bound, fp64 re-evaluation, and the lanes' private bests are
// merged at the end by (d2, index).  Groups of one warp run different numbers of steps; every warp-level primitive is
// called with the group's own lane mask.
#define PC_COOP_WARPS 4
#define PC_COOP_CAP(G) (32 * (G))          // frontier entries per group: 8 KB of shared memory per warp for every G

template <int KIND, int G>
__global__ void __launch_bounds__(32 * PC_COOP_WARPS)
pc_query_coop_kernel(pc_tree T, pc_radius_dev R, const float *__restrict__ q, int64_t m, int qstride,
                     int32_t *__restrict__ out_idx, float *__restrict__ out_f)
{
    constexpr int GROUPS = 32 / G, CAP = PC_COOP_CAP(G);
    static_assert(CAP >= 2 * G + PC_STACK + 8, "frontier too small for the depth-first fallback");
    __shared__ uint2 s_front[PC_COOP_WARPS * GROUPS][CAP];      // (inner node, float bits of its box distance)
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int gl = lane & (G - 1), grp = lane / G;              // lane inside the group, group inside the warp
    const uint32_t gmask = G == 32 ? PC_FULL_MASK : (((1u << G) - 1u) << (grp * G));
    const int64_t k = ((int64_t)blockIdx.x * PC_COOP_WARPS + w) * GROUPS + grp;
    if (k >= m) return;
    const float *qq = q + (size_t)k * qstride;
    const float qv[1][3] = { { qq[0], qq[1], qq[2] } };
    const float qx = qv[0][0], qy = qv[0][1], qz = qv[0][2];
    bool search = T.n_points > 0;
    if (KIND == PC_KIND_RADIUS && search && pc_radius_early_out((double)qx, (double)qy, (double)qz, R)) search = false;
    if (!search) { if (gl == 0) pc_write_trivial<KIND>(R, (uint32_t)k, out_idx, out_f); return; }
    pc_best b[1];
    b[0].d2 = INFINITY; b[0].idx = -1; b[0].thr = (KIND == PC_KIND_RADIUS) ? R.bound_thr : FLT_MAX;
    uint2 *F = s_front[w * GROUPS + grp];
    // start from the seeds: the top of the tree already expanded to <= 32 inner nodes (box distance unknown: 0), the few
    // leaves met on the way scanned by the first lanes
    const int n_seed = (int)T.seeds[0], n_seed_leaf = (int)T.seeds[1];
    for (int j = gl; j < n_seed_leaf; j += G) pc_scan_leaf<1>(T.points + (T.seeds[PC_SEED_LEAF + 2 * j] & ~PC_REF_LEAF), qv, b);
    for (int j = gl; j < n_seed; j += G) F[j] = make_uint2(T.seeds[PC_SEED_INNER + j], 0u);
    int size = n_seed;
    __syncwarp(gmask);
    const uint32_t lt = (1u << gl) - 1u;
    while (size > 0) {
        // take the top of the frontier, one node per lane (grows it by at most G entries); close to the capacity fall back
        // to one node per step -- a plain DFS, which adds at most one entry per tree level (<= PC_STACK)
        const int take = (size + G + PC_STACK <= CAP) ? min(size, G) : 1;
        bool active = gl < take;
        uint2 e = make_uint2(0u, 0u);
        if (active) e = F[size - 1 - gl];
        size -= take;
        __syncwarp(gmask);
        active = active && __uint_as_float(e.y) <= b[0].thr;
        float dn = INFINITY, df = INFINITY;      // inner children to push (INFINITY: none)
        uint32_t cn = 0, cf = 0;
        if (active) {
            const pc_rec rec = pc_load_rec(T.rec + 4ull * e.x);
            const float2 dd = pc_rec_d2(rec, qx, qy, qz);
            const float d0 = dd.x, d1 = dd.y;
            const uint32_t r0 = pc_rec_ref(rec, 0), r1 = pc_rec_ref(rec, 1);
            const bool first0 = d0 <= d1;
            const uint32_t rn = first0 ? r0 : r1, rf = first0 ? r1 : r0;
            const float dnn = fminf(d0, d1), dff = fmaxf(d0, d1);
            if (dnn <= b[0].thr) {
                if (rn & PC_REF_LEAF) pc_scan_leaf<1>(T.points + (rn & ~PC_REF_LEAF), qv, b);
                else { cn = rn; dn = dnn; }
            }
            if (dff <= b[0].thr) {
                if (rf & PC_REF_LEAF) pc_scan_leaf<1>(T.points + (rf & ~PC_REF_LEAF), qv, b);
                else { cf = rf; df = dff; }
            }
        }
        // one bound for the whole group (thr >= 0, so the float order is the order of its bits)
        b[0].thr = __uint_as_float(__reduce_min_sync(gmask, __float_as_uint(b[0].thr)));
        const bool wn = dn <= b[0].thr, wf = df <= b[0].thr;
        const uint32_t mf = (__ballot_sync(gmask, wf) & gmask) >> (grp * G), mn = (__ballot_sync(gmask, wn) & gmask) >> (grp * G);
        const int nf = __popc(mf), nn = __popc(mn);
        if (wf) F[size + __popc(mf & lt)] = make_uint2(cf, __float_as_uint(df));
        if (wn) F[size + nf + (nn - 1 - __popc(mn & lt))] = make_uint2(cn, __float_as_uint(dn));   // lane 0's child ends on top
        size += nf + nn;
        __syncwarp(gmask);
    }
    // merge the lanes' private bests: smallest (d2, index); d2 >= 0, so its bit pattern orders like the value
    long long key = __double_as_longlong(b[0].d2);
    uint32_t id = (uint32_t)b[0].idx;
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
        const long long k2 = __shfl_xor_sync(gmask, key, o);
        const uint32_t i2 = __shfl_xor_sync(gmask, id, o);
        if (k2 < key || (k2 == key && i2 < id)) { key = k2; id = i2; }
    }
    if (gl == 0) {
        b[0].d2 = __longlong_as_double(key); b[0].idx = (int32_t)id;
        pc_write_result<KIND>(R, b[0], (uint32_t)k, out_idx, out_f);
    }
}

// ---- ordering pass of a batch --------------------------------------------------------------------------
// Hilbert key of every query in the index's frame (top `30 - drop_bits` bits), so that the lanes of a warp walk the
// same part of the tree.  For radius batches the sensing-range early-out (corridor_finder.cpp:115-116) is evaluated
// here, once, coalesced: such queries get their result now; the others are compacted into (key, slot) pairs and
// n_search counts them -- only those are sorted and searched.
//
// pc_batch_shard: the cubic cells of the curve's frame at a batch-dependent level are dealt to the ranks by a hash of the
// cell coordinates; a query that another rank owns is dropped right after its 12 bytes were read (no early-out test, no
// curve key), so the pass over the full batch that every rank makes stays cheap.  A
// rank's share is then as dense in space as the whole batch (dense packets) and spread over the whole map (equal cost per
// rank).  The level is computed HERE, from the index's bounding box, the batch size and the number of ranks only -- all
// identical on every rank that holds a replica -- so all ranks agree on the owner of every query whatever the state of their
// host-side caches: the finest cells (<= 1024 per axis) that still hold >= 1024 queries each, refined (down to 128 queries
// per cell) while a rank would get fewer than 256 of them.  Finer cells balance the ranks better, coarser ones cut fewer
// packets at a cell's end, where the next query of the share lies some cells away (C5 on 8 ranks, cells of 735 / 5 880 /
// 47 000 queries: 6.85 / 6.43 / 6.45 ms for the slowest rank, shares 12.3-12.7 / 12.1-12.8 / 11.5-13.1 % of the batch).
// Measured on C5 with 8 GPUs: array slices 37 ms; contiguous stretches of the curve 41 ms and round-robin 32^3 cells 43 ms
// (both unbalanced: 18..42 ms per rank -- on a flat map the low bits of the cell index encode the z layer); hashed cells:
// profiles/r1_c5_strong_scaling.jsonl.
#ifndef PC_SHARD_CELL_QUERIES
#define PC_SHARD_CELL_QUERIES 1024     // queries a cell of the share grid should hold (16 packets: one in 16 is cut by the cell's end)
#endif
#define PC_SHARD_CELL_MIN_QUERIES 128  // ... and never fewer than this
#define PC_SHARD_CELLS_PER_RANK 256    // cells a rank should own at least (balance: the shares differ by ~ 1 / sqrt(cells))
__device__ __forceinline__ int pc_shard_level(const uint32_t *__restrict__ bbox, int64_t m, int shard_n)
{
    float ext[3], emax = 0.f;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        ext[a] = pc_ordered_to_float(bbox[3 + a]) - pc_ordered_to_float(bbox[a]);
        emax = fmaxf(emax, ext[a]);
    }
    if (!(emax > 0.f) || !(emax < INFINITY)) return 2;
    // queries per cell at level lv (2^lv cells per axis of the cubic frame; the batch is taken to fill the bounding box)
    auto per_cell = [&](int lv, double *cells) {
        const double c = (double)emax / (double)(1 << lv);
        double v = 1.0;
#pragma unroll
        for (int a = 0; a < 3; a++) v *= (double)ext[a] > c ? (double)ext[a] : c;
        *cells = v / (c * c * c);
        return (double)m / *cells;
    };
    int lv = 2;
    double cells = 0.0;
    for (int l = 10; l > 2; l--)
        if (per_cell(l, &cells) >= (double)PC_SHARD_CELL_QUERIES) { lv = l; break; }
    // too few cells to deal out evenly: finer ones, as long as they still hold a couple of packets
    while (lv < 10) {
        per_cell(lv, &cells);
        if (cells >= (double)PC_SHARD_CELLS_PER_RANK * shard_n) break;
        if (per_cell(lv + 1, &cells) < (double)PC_SHARD_CELL_MIN_QUERIES) break;
        lv++;
    }
    return lv;
}

#define PC_KEY_ITEMS 8          // queries per thread and round of the key kernel: eight loads in flight, one atomic per 2048 queries

// pc_batch_shard: the rank that owns a cell of the index's cubic frame (cell coordinates at 10 bits per axis, `sh` low bits
// dropped): a murmur-style finaliser of the packed coordinates, mapped to [0, shard_n) by a multiply-shift (no division)
__device__ __forceinline__ int pc_shard_owner(uint32_t cx, uint32_t cy, uint32_t cz, int sh, int shard_n)
{
    uint32_t h = (cx >> sh) | ((cy >> sh) << 10) | ((cz >> sh) << 20);
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    return (int)__umulhi(h, (uint32_t)shard_n);
}

// pc_batch_shard, first half of a round of the key / bin-count kernels: which of the CTA's 256 x PC_KEY_ITEMS queries does this
// rank own?  The batch is in arbitrary order, so the owned queries (1 / shard_n of them) are scattered over all lanes: running
// the expensive part of the pass (early-out test in fp64, curve key) in place would cost every warp the full instruction count
// with a few lanes active -- measured: 845 M warp instructions for a rank's pass over 8 x 10^7 queries, 10 of 32 lanes active,
// as slow as keying the whole batch.  So the owned queries are compacted into shared memory (x, y, z, slot) and handed back
// densely, entry j * 256 + thread: the rest of the round runs on full warps and costs in proportion to the share.
// Returns the number of owned queries; x / y / z / slot / have are rewritten.  Two barriers; s_warp is free again afterwards.
__device__ __forceinline__ uint32_t pc_shard_compact(float (&x)[PC_KEY_ITEMS], float (&y)[PC_KEY_ITEMS], float (&z)[PC_KEY_ITEMS],
                                                     uint32_t (&slot)[PC_KEY_ITEMS], bool (&have)[PC_KEY_ITEMS], const pc_frame &f, int sh,
                                                     int shard_rank, int shard_n, float4 *s_list, uint32_t *s_warp)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t lt = pc_lanemask_lt();
    uint32_t om[PC_KEY_ITEMS], warp_total = 0;
#pragma unroll
    for (int j = 0; j < PC_KEY_ITEMS; j++) {
        bool own = have[j];
        if (own) {
            const uint32_t cx = pc_cell_coord(x[j], f.lo[0], f.inv_cell, f.max_cell), cy = pc_cell_coord(y[j], f.lo[1], f.inv_cell, f.max_cell),
                           cz = pc_cell_coord(z[j], f.lo[2], f.inv_cell, f.max_cell);
            own = pc_shard_owner(cx, cy, cz, sh, shard_n) == shard_rank;
        }
        om[j] = __ballot_sync(PC_FULL_MASK, own);
        warp_total += __popc(om[j]);
    }
    if (lane == 0) s_warp[warp] = warp_total;
    __syncthreads();
    uint32_t off = 0, count = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) { const uint32_t t = s_warp[w]; if (w < warp) off += t; count += t; }
#pragma unroll
    for (int j = 0; j < PC_KEY_ITEMS; j++) {
        if ((om[j] >> lane) & 1u) s_list[off + __popc(om[j] & lt)] = make_float4(x[j], y[j], z[j], __uint_as_float(slot[j]));
        off += __popc(om[j]);
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < PC_KEY_ITEMS; j++) {
        const uint32_t e = (uint32_t)j * 256u + threadIdx.x;
        have[j] = e < count;
        if (have[j]) { const float4 v = s_list[e]; x[j] = v.x; y[j] = v.y; z[j] = v.z; slot[j] = __float_as_uint(v.w); }
    }
    return count;
}

template <int KIND, bool SHARDED>
__global__ void __launch_bounds__(256)
pc_query_key_kernel(const float *__restrict__ q, int64_t m, int qstride, const uint32_t *__restrict__ bbox, int drop_bits,
                    pc_radius_dev R, int32_t *__restrict__ out_idx, float *__restrict__ out_f,
                    uint32_t *__restrict__ keys, uint32_t *__restrict__ vals, unsigned long long *__restrict__ n_search,
                    int shard_rank, int shard_n, uint32_t *__restrict__ ghist, int hist_passes)
{
    // ghist (nullable): digit histograms of the hist_passes 8-bit passes that will sort the compacted keys (radix_sort.cuh,
    // onesweep path) -- counted here, while the key is in a register, instead of by a separate pass over the keys.  The
    // grid is one wave of CTAs, each striding over the batch in rounds of 256 x PC_KEY_ITEMS queries, so that a CTA flushes
    // its histograms to global memory once and reserves its output range with one atomic per round.
    __shared__ uint32_t s_hist[4][RS_RADIX];
    __shared__ uint32_t s_warp[8];
    __shared__ unsigned long long s_base;
    __shared__ int s_shard_shift;
    __shared__ float4 s_list[SHARDED ? 256 * PC_KEY_ITEMS : 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t lt = pc_lanemask_lt();
    if (ghist) for (int j = threadIdx.x; j < hist_passes * RS_RADIX; j += 256) (&s_hist[0][0])[j] = 0;
    if (SHARDED && threadIdx.x == 0) s_shard_shift = 10 - pc_shard_level(bbox, m, shard_n);      // cell coordinate bits dropped per axis
    __syncthreads();
    const pc_frame f = pc_make_frame(bbox, 10);
    const int sh = SHARDED ? s_shard_shift : 0;
    for (int64_t base = (int64_t)blockIdx.x * (256 * PC_KEY_ITEMS); base < m; base += (int64_t)gridDim.x * (256 * PC_KEY_ITEMS)) {
        float x[PC_KEY_ITEMS], y[PC_KEY_ITEMS], z[PC_KEY_ITEMS];
        uint32_t slot[PC_KEY_ITEMS];
        bool have[PC_KEY_ITEMS];
#pragma unroll
        for (int j = 0; j < PC_KEY_ITEMS; j++) {
            const int64_t i = base + j * 256 + threadIdx.x;
            have[j] = i < m;
            slot[j] = (uint32_t)i;
            if (have[j]) { const float *p = q + i * qstride; x[j] = p[0]; y[j] = p[1]; z[j] = p[2]; }
            else x[j] = y[j] = z[j] = 0.f;
        }
        if (SHARDED) pc_shard_compact(x, y, z, slot, have, f, sh, shard_rank, shard_n, s_list, s_warp);
        uint32_t key[PC_KEY_ITEMS], mask[PC_KEY_ITEMS];
        uint32_t warp_total = 0;
#pragma unroll
        for (int j = 0; j < PC_KEY_ITEMS; j++) {
            bool search = have[j];
            key[j] = 0;
            if (search) {
                if (KIND == PC_KIND_RADIUS && pc_radius_early_out((double)x[j], (double)y[j], (double)z[j], R)) {
                    search = false;
                    pc_write_trivial<KIND>(R, slot[j], out_idx, out_f);
                } else {
                    const uint32_t cx = pc_cell_coord(x[j], f.lo[0], f.inv_cell, f.max_cell), cy = pc_cell_coord(y[j], f.lo[1], f.inv_cell, f.max_cell),
                                   cz = pc_cell_coord(z[j], f.lo[2], f.inv_cell, f.max_cell);
                    key[j] = pc_hilbert30_cells(cx, cy, cz) >> drop_bits;
                }
            }
            mask[j] = __ballot_sync(PC_FULL_MASK, search);
            warp_total += __popc(mask[j]);
        }
        // compact the queries that still need a search: only those are sorted and searched.  The slot a query lands in depends
        // on CTA scheduling, which changes the composition of packets but never a result.
        if (lane == 0) s_warp[warp] = warp_total;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tot = 0;
            for (int w = 0; w < 8; w++) { const uint32_t c = s_warp[w]; s_warp[w] = tot; tot += c; }
            s_base = tot ? atomicAdd(n_search, (unsigned long long)tot) : 0ull;
        }
        __syncthreads();
        unsigned long long pos = s_base + s_warp[warp];
#pragma unroll
        for (int j = 0; j < PC_KEY_ITEMS; j++) {
            if ((mask[j] >> lane) & 1u) {
                const unsigned long long p = pos + __popc(mask[j] & lt);
                keys[p] = key[j];
                vals[p] = slot[j];
                if (ghist) for (int h = 0; h < hist_passes; h++) atomicAdd(&s_hist[h][(key[j] >> (8 * h)) & (RS_RADIX - 1)], 1u);
            }
            pos += __popc(mask[j]);
        }
        __syncthreads();            // s_warp / s_base are rewritten by the next round
    }
    if (ghist) {
        __syncthreads();
        for (int j = threadIdx.x; j < hist_passes * RS_RADIX; j += 256) {
            const uint32_t c = (&s_hist[0][0])[j];
            if (c) atomicAdd(&ghist[j], c);
        }
    }
}

// ---- ordering pass, cell-binning variant ---------------------------------------------------------------------------------
// A batch only has to be GROUPED by small cells -- which queries share a packet matters, their order inside it does not.  So
// instead of radix-sorting (key, slot) pairs, the batch is counting-sorted by a 21-bit cell id in one histogram pass and one
// scatter pass, and the scatter writes the queries themselves, (x, y, z, slot) as float4, so that the search kernel reads its
// input coalesced.  The 2^21 cells are cubes of one edge h fitted to the cloud's bounding BOX, not its bounding cube (a flat map
// of 77 x 77 x 8 m gets 0.3 m cells -- 8 + 8 + 5 bits -- where a cubic frame of 7 bits per axis gives 0.6 m ones, which cost the
// search 12 %): cell id = (block of 2^b x 2^b x 2^b cells, row-major over the blocks) . (3-D Hilbert index inside the block),
// b = the smallest per-axis bit count:
//   pc_bin_count_kernel    cell of every query; sensing-range early-outs answered on the spot; count per cell (red.global)
//   pc_bin_scan_*          exclusive scan of the 2^21 counts (three small kernels); the total = number of queries to search
//   pc_bin_scatter_kernel  position = atomicAdd(cursor[cell]) -- the order inside a cell is whatever the atomics give
// Used when a cell holds at most a few packets (the density test that picked the 24-bit radix sort); denser batches keep the
// radix sort on the full 30-bit key, whose order inside a coarse cell matters.
#define PC_BIN_MAX_BITS 24              // most cells a batch is binned into: 2^24 (the count follows the batch size, see pc_index.cu)
#define PC_BIN_SKIP 0xffffffffu
#define PC_BIN_SCAN_TILE 2048            // bins per CTA of the scan kernels (256 threads x 8)

// the frame of the binning grid, derived from the index's bounding box on the device (identical on every rank)
struct pc_bin_frame {
    float lo[3], inv_h;
    int bits[3];          // cells per axis = 2^bits, sum <= total_bits
    int low;              // min(bits): the 3-D Hilbert index covers the low `low` bits of every axis
    int sh_y, sh_z;       // block index = hx | hy << sh_y | hz << sh_z, h = the axis' bits above `low` (row-major over the blocks:
                          // with <= a few hundred blocks of 2^low cells per axis their order hardly matters)
};

__device__ __forceinline__ pc_bin_frame pc_make_bin_frame(const uint32_t *__restrict__ bbox, int total_bits)
{
    pc_bin_frame F;
    float ext[3], emax = 0.f;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        F.lo[a] = pc_ordered_to_float(bbox[a]);
        ext[a] = pc_ordered_to_float(bbox[3 + a]) - F.lo[a];
        if (!(ext[a] >= 0.f) || !(ext[a] < INFINITY)) ext[a] = 0.f;
        emax = fmaxf(emax, ext[a]);
    }
    if (!(emax > 0.f)) { F.inv_h = 0.f; F.bits[0] = F.bits[1] = F.bits[2] = F.low = 1; F.sh_y = F.sh_z = 0; return F; }
    // smallest h (in steps of 2^(1/3)) whose per-axis power-of-two cell counts fit total_bits bits
    float vol = 1.f;
#pragma unroll
    for (int a = 0; a < 3; a++) vol *= fmaxf(ext[a], emax * (1.0f / 1024.0f));
    float h = cbrtf(vol / (float)(1u << total_bits));
    for (int it = 0; it < 64; it++) {
        int sum = 0;
#pragma unroll
        for (int a = 0; a < 3; a++) {
            int b = 1;
            while (b < 10 && (float)(1 << b) * h <= ext[a] * 1.0001f) b++;
            F.bits[a] = b; sum += b;
        }
        if (sum <= total_bits && (float)(1 << F.bits[0]) * h > ext[0] && (float)(1 << F.bits[1]) * h > ext[1] && (float)(1 << F.bits[2]) * h > ext[2]) break;
        h *= 1.2599211f;
    }
    F.inv_h = 1.0f / h;
    F.low = min(F.bits[0], min(F.bits[1], F.bits[2]));
    F.sh_y = F.bits[0] - F.low;
    F.sh_z = F.sh_y + F.bits[1] - F.low;
    return F;
}

__device__ __forceinline__ uint32_t pc_hilbert_cells_var(uint32_t x, uint32_t y, uint32_t z, int bits);
template <int BITS> __device__ __forceinline__ uint32_t pc_hilbert_cells_n(uint32_t x, uint32_t y, uint32_t z);

// 3-D Hilbert indices of the 16^3 and 32^3 blocks as lookup tables (2 + 64 KB, L1-resident): the transform itself is ~100
// instructions per query, most of what the count kernel executes.  Filled once per device by pc_hilbert_lut_kernel.
#define PC_LUT4_WORDS 4096
#define PC_LUT5_WORDS 32768
__global__ void __launch_bounds__(256)
pc_hilbert_lut_kernel(uint16_t *__restrict__ lut4, uint16_t *__restrict__ lut5);

__device__ __forceinline__ uint32_t pc_bin_of(float x, float y, float z, const pc_bin_frame &F, const uint16_t *__restrict__ lut)
{
    uint32_t c[3];
    const float v[3] = { x, y, z };
#pragma unroll
    for (int a = 0; a < 3; a++) {
        float t = (v[a] - F.lo[a]) * F.inv_h;
        t = fminf(fmaxf(t, 0.0f), (float)((1 << F.bits[a]) - 1));      // NaN -> 0; queries outside the cloud's box -> border cells
        c[a] = (uint32_t)t;
    }
    const uint32_t mask = (1u << F.low) - 1u;
    uint32_t inner;                                       // unrolled transforms for the usual block sizes (warp-uniform switch)
    switch (F.low) {
    case 4: inner = __ldg(lut + (((c[2] & mask) << 8) | ((c[1] & mask) << 4) | (c[0] & mask))); break;
    case 5: inner = __ldg(lut + PC_LUT4_WORDS + (((c[2] & mask) << 10) | ((c[1] & mask) << 5) | (c[0] & mask))); break;
    case 6: inner = pc_hilbert_cells_n<6>(c[0] & mask, c[1] & mask, c[2] & mask); break;
    case 7: inner = pc_hilbert_cells_n<7>(c[0] & mask, c[1] & mask, c[2] & mask); break;
    default: inner = pc_hilbert_cells_var(c[0] & mask, c[1] & mask, c[2] & mask, F.low); break;
    }
    const uint32_t blk = (c[0] >> F.low) | ((c[1] >> F.low) << F.sh_y) | ((c[2] >> F.low) << F.sh_z);
    return (blk << (3 * F.low)) | inner;
}

// Skilling's transform for a runtime number of bits per axis (1..10)
__device__ __forceinline__ uint32_t pc_hilbert_cells_var(uint32_t x, uint32_t y, uint32_t z, int bits)
{
    uint32_t X[3] = { x, y, z };
    const uint32_t M = 1u << (bits - 1);
    for (uint32_t Q = M; Q > 1; Q >>= 1) {
        const uint32_t P = Q - 1;
#pragma unroll
        for (int i = 0; i < 3; i++) {
            if (X[i] & Q) X[0] ^= P;
            else { const uint32_t t = (X[0] ^ X[i]) & P; X[0] ^= t; X[i] ^= t; }
        }
    }
    X[1] ^= X[0];
    X[2] ^= X[1];
    uint32_t t = 0;
    for (uint32_t Q = M; Q > 1; Q >>= 1) if (X[2] & Q) t ^= Q - 1;
    X[0] ^= t; X[1] ^= t; X[2] ^= t;
    return (pc_spread10(X[0]) << 2) | (pc_spread10(X[1]) << 1) | pc_spread10(X[2]);
}

// Skilling's transform for BITS bits per axis (compile-time)
template <int BITS>
__device__ __forceinline__ uint32_t pc_hilbert_cells_n(uint32_t x, uint32_t y, uint32_t z)
{
    uint32_t X[3] = { x, y, z };
    const uint32_t M = 1u << (BITS - 1);
#pragma unroll
    for (uint32_t Q = M; Q > 1; Q >>= 1) {
        const uint32_t P = Q - 1;
#pragma unroll
        for (int i = 0; i < 3; i++) {
            if (X[i] & Q) X[0] ^= P;
            else { const uint32_t t = (X[0] ^ X[i]) & P; X[0] ^= t; X[i] ^= t; }
        }
    }
    X[1] ^= X[0];
    X[2] ^= X[1];
    uint32_t t = 0;
#pragma unroll
    for (uint32_t Q = M; Q > 1; Q >>= 1) if (X[2] & Q) t ^= Q - 1;
    X[0] ^= t; X[1] ^= t; X[2] ^= t;
    return (pc_spread10(X[0]) << 2) | (pc_spread10(X[1]) << 1) | pc_spread10(X[2]);
}

__global__ void __launch_bounds__(256)
pc_hilbert_lut_kernel(uint16_t *__restrict__ lut4, uint16_t *__restrict__ lut5)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < PC_LUT4_WORDS) lut4[i] = (uint16_t)pc_hilbert_cells_n<4>(i & 15u, (i >> 4) & 15u, (i >> 8) & 15u);
    if (i < PC_LUT5_WORDS) lut5[i] = (uint16_t)pc_hilbert_cells_n<5>(i & 31u, (i >> 5) & 31u, (i >> 10) & 31u);
}

template <int KIND, bool SHARDED>
__global__ void __launch_bounds__(256)
pc_bin_count_kernel(const float *__restrict__ q, int64_t m, int qstride, const uint32_t *__restrict__ bbox,
                    pc_radius_dev R, int32_t *__restrict__ out_idx, float *__restrict__ out_f,
                    uint32_t *__restrict__ cellkey, uint32_t *__restrict__ bins, int bin_bits, int shard_rank, int shard_n,
                    const uint16_t *__restrict__ lut)
{
    __shared__ int s_shard_shift;
    __shared__ pc_bin_frame s_frame;
    __shared__ uint32_t s_warp[8];
    __shared__ float4 s_list[SHARDED ? 256 * PC_KEY_ITEMS : 1];
    if (threadIdx.x == 0) {
        s_frame = pc_make_bin_frame(bbox, bin_bits);
        if (SHARDED) s_shard_shift = 10 - pc_shard_level(bbox, m, shard_n);
    }
    __syncthreads();
    const pc_bin_frame F = s_frame;
    const pc_frame f = pc_make_frame(bbox, 10);
    const int sh = SHARDED ? s_shard_shift : 0;
    for (int64_t base = (int64_t)blockIdx.x * (256 * PC_KEY_ITEMS); base < m; base += (int64_t)gridDim.x * (256 * PC_KEY_ITEMS)) {
        float x[PC_KEY_ITEMS], y[PC_KEY_ITEMS], z[PC_KEY_ITEMS];
        uint32_t slot[PC_KEY_ITEMS];
        bool have[PC_KEY_ITEMS];
#pragma unroll
        for (int j = 0; j < PC_KEY_ITEMS; j++) {
            const int64_t i = base + j * 256 + threadIdx.x;
            have[j] = i < m;
            slot[j] = (uint32_t)i;
            if (have[j]) { const float *p = q + i * qstride; x[j] = __ldcs(p); y[j] = __ldcs(p + 1); z[j] = __ldcs(p + 2); }   // read once: evict first
            else x[j] = y[j] = z[j] = 0.f;
        }
        if (SHARDED) {
            // every query's cell key is written (the scatter pass reads them all): "skip" for the whole round here, coalesced;
            // the owned queries overwrite theirs below, after the barriers of the compaction
#pragma unroll
            for (int j = 0; j < PC_KEY_ITEMS; j++)
                if (have[j]) cellkey[slot[j]] = PC_BIN_SKIP;
            pc_shard_compact(x, y, z, slot, have, f, sh, shard_rank, shard_n, s_list, s_warp);
        }
#pragma unroll
        for (int j = 0; j < PC_KEY_ITEMS; j++) {
            if (!have[j]) continue;
            bool search = true;
            if (KIND == PC_KIND_RADIUS && pc_radius_early_out((double)x[j], (double)y[j], (double)z[j], R)) {
                search = false;
                pc_write_trivial<KIND>(R, slot[j], out_idx, out_f);
            }
            uint32_t key = PC_BIN_SKIP;
            if (search) {
                key = pc_bin_of(x[j], y[j], z[j], F, lut);
                atomicAdd(bins + key, 1u);
            }
            if (!SHARDED || search) cellkey[slot[j]] = key;
        }
    }
}

// exclusive scan of n_bins counts in place: tile sums -> scan of the tile sums by one CTA (total -> *n_search) -> apply
__global__ void __launch_bounds__(256)
pc_bin_scan_tiles(const uint32_t *__restrict__ bins, uint32_t *__restrict__ tile_sum)
{
    __shared__ uint32_t s_w[8];
    const uint4 *p = reinterpret_cast<const uint4 *>(bins + (size_t)blockIdx.x * PC_BIN_SCAN_TILE) + 2 * threadIdx.x;
    const uint4 a = p[0], b = p[1];
    uint32_t v = a.x + a.y + a.z + a.w + b.x + b.y + b.z + b.w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(PC_FULL_MASK, v, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < 8; w++) t += s_w[w]; tile_sum[blockIdx.x] = t; }
}

__global__ void __launch_bounds__(1024)
pc_bin_scan_top(uint32_t *__restrict__ tile_sum, int n_tiles, unsigned long long *__restrict__ n_search)
{
    __shared__ uint32_t s_w[32];
    __shared__ uint32_t s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < n_tiles; base += 1024) {
        const int i = base + threadIdx.x;
        const uint32_t v = i < n_tiles ? tile_sum[i] : 0u;
        uint32_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(PC_FULL_MASK, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) s_w[warp] = incl;
        __syncthreads();
        uint32_t woff = 0;
        for (int w = 0; w < warp; w++) woff += s_w[w];
        const uint32_t carry = s_carry;
        if (i < n_tiles) tile_sum[i] = carry + woff + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + woff + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_search = (unsigned long long)s_carry;
}

__global__ void __launch_bounds__(256)
pc_bin_scan_apply(uint32_t *__restrict__ bins, const uint32_t *__restrict__ tile_sum)
{
    __shared__ uint32_t s_w[8];
    uint4 *p = reinterpret_cast<uint4 *>(bins + (size_t)blockIdx.x * PC_BIN_SCAN_TILE) + 2 * threadIdx.x;
    uint4 a = p[0], b = p[1];
    const uint32_t mine = a.x + a.y + a.z + a.w + b.x + b.y + b.z + b.w;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(PC_FULL_MASK, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    uint32_t run = tile_sum[blockIdx.x] + incl - mine;
    for (int w = 0; w < warp; w++) run += s_w[w];
    uint32_t t;
    t = a.x; a.x = run; run += t;  t = a.y; a.y = run; run += t;  t = a.z; a.z = run; run += t;  t = a.w; a.w = run; run += t;
    t = b.x; b.x = run; run += t;  t = b.y; b.y = run; run += t;  t = b.z; b.z = run; run += t;  t = b.w; b.w = run; run += t;
    p[0] = a; p[1] = b;
}

// OWNED_ONLY (pc_batch_shard): most queries belong to other ranks -- their coordinates are not read again; otherwise the
// coordinate loads are issued together with the key loads (one round trip instead of two).
template <bool OWNED_ONLY>
__global__ void __launch_bounds__(256)
pc_bin_scatter_kernel(const float *__restrict__ q, int64_t m, int qstride, const uint32_t *__restrict__ cellkey,
                      uint32_t *__restrict__ cursor, float4 *__restrict__ ordered)
{
    for (int64_t base = (int64_t)blockIdx.x * (256 * PC_KEY_ITEMS); base < m; base += (int64_t)gridDim.x * (256 * PC_KEY_ITEMS)) {
        float x[PC_KEY_ITEMS], y[PC_KEY_ITEMS], z[PC_KEY_ITEMS];
        uint32_t key[PC_KEY_ITEMS];
#pragma unroll
        for (int j = 0; j < PC_KEY_ITEMS; j++) {
            const int64_t i = base + j * 256 + threadIdx.x;
            key[j] = PC_BIN_SKIP;
            if (OWNED_ONLY) x[j] = y[j] = z[j] = 0.f;
            if (i < m) {
                key[j] = __ldcs(cellkey + i);
                if (!OWNED_ONLY) { const float *p = q + i * qstride; x[j] = __ldcs(p); y[j] = __ldcs(p + 1); z[j] = __ldcs(p + 2); }
            }
        }
        if (OWNED_ONLY) {
#pragma unroll
            for (int j = 0; j < PC_KEY_ITEMS; j++)
                if (key[j] != PC_BIN_SKIP) { const float *p = q + (base + j * 256 + threadIdx.x) * qstride; x[j] = __ldcs(p); y[j] = __ldcs(p + 1); z[j] = __ldcs(p + 2); }
        }
        // all of a thread's cursor atomics first, then the stores: eight round trips in flight instead of eight in a row
        uint32_t pos[PC_KEY_ITEMS];
#pragma unroll
        for (int j = 0; j < PC_KEY_ITEMS; j++) {
            pos[j] = 0;
            if (key[j] != PC_BIN_SKIP) pos[j] = atomicAdd(cursor + key[j], 1u);
        }
#pragma unroll
        for (int j = 0; j < PC_KEY_ITEMS; j++)
            if (key[j] != PC_BIN_SKIP) ordered[pos[j]] = make_float4(x[j], y[j], z[j], __uint_as_float((uint32_t)(base + j * 256 + threadIdx.x)));
    }
}
