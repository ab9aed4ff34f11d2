// range_kernels.cuh -- fixed-radius range queries: all points with d2 <= range^2.
//
// Replaces find_nearest / kd_nearest_range3 (Utils/kdtree/src/kdtree.c:262-293,595-602) and the kd_res_*
// iteration (kdtree.c:613-650).  The hit test is the reference's inclusive `dist_sq <= SQ(range)` (kdtree.c:273)
// evaluated in fp64 in its operation order; unlike the reference the far side of a split is never skipped, so a
// point at exactly `range` is always reported (the reference misses it from one side, kdtree.c:283 -- SURVEY 8c-5).
// One WARP per query.  The walk runs ONCE for almost every query: the counting pass also captures the hits of lists up to
// PC_RCAP_HITS entries in shared memory, sorts them by original index there and parks them in a staging buffer (one
// atomicAdd per query for the place); after the scan of the counts a copy kernel moves every parked list to its CSR
// position.  Only lists longer than that are walked a second time (fill pass, given their offsets).  A call that asks for
// the offsets only runs the plain counting pass.
#pragma once
#include "query_kernels.cuh"

// in-place heap sort of one query's list (ascending original index); lists are short (tens to hundreds)
__device__ __forceinline__ void pc_sort_list(int32_t *__restrict__ a, int64_t n)
{
    if (n < 2) return;
    for (int64_t start = n / 2 - 1; start >= 0; start--) {
        int64_t root = start;
        for (;;) {
            int64_t child = 2 * root + 1;
            if (child >= n) break;
            if (child + 1 < n && a[child] < a[child + 1]) child++;
            if (a[root] >= a[child]) break;
            int32_t t = a[root]; a[root] = a[child]; a[child] = t;
            root = child;
        }
    }
    for (int64_t end = n - 1; end > 0; end--) {
        int32_t t = a[0]; a[0] = a[end]; a[end] = t;
        int64_t root = 0;
        for (;;) {
            int64_t child = 2 * root + 1;
            if (child >= end) break;
            if (child + 1 < end && a[child] < a[child + 1]) child++;
            if (a[root] >= a[child]) break;
            int32_t u = a[root]; a[root] = a[child]; a[child] = u;
            root = child;
        }
    }
}

// ---- one WARP per range query -----------------------------------------------------------------------------------------
// Same frontier walk as pc_query_coop_kernel (query_kernels.cuh), without a bound to tighten (pc_range_walk below); the hits
// are appended at ballot-computed positions.  The count / capture pass and the fill pass are the same walk; the fill pass
// then sorts its list by original index with a bitonic network in the same shared memory (lists up to 1024 hits);
// longer lists are queued and sorted afterwards by pc_range_sort_long_kernel, one CTA per list (up to 32768 hits in shared
// memory; beyond that a single-thread heap sort -- a query that returns more than that is a job for pc_sphere_gather).
#define PC_RCOOP_CAP 1024
#define PC_RCOOP_WARPS 4
#define PC_RCAP_HITS 512         // lists up to this length are captured by the counting pass (C1: 99.9 % of them)
#ifndef PC_RCAP_MIN_CTAS
#define PC_RCAP_MIN_CTAS 8       // resident CTAs per SM the capturing pass is compiled for (64 registers).  C1 range batch: 7 CTAs
                                 // (66 registers, no spill) 0.93 ms, 8: 0.80, 9: 0.93, 10 (48 registers): 1.01, 12: 1.13
#endif
#define PC_RFILL_WARP_SORT 256   // fill pass: longer lists are sorted by a whole CTA each (pc_range_sort_long_kernel) -- a 1024-entry
                                 // bitonic network run by ONE warp was a 100 us tail for a handful of lists
#define PC_RANGE_COUNT 0
#define PC_RANGE_FILL 1
#define PC_RANGE_CAPTURE 2

// bitonic sort of N (power of two >= 32) words in a warp's shared memory
__device__ __forceinline__ void pc_warp_bitonic(uint32_t *F, int N, int lane)
{
    for (int k2 = 2; k2 <= N; k2 <<= 1) {
        for (int j = k2 >> 1; j > 0; j >>= 1) {
            for (int t = lane; t < (N >> 1); t += 32) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), l = i | j;
                const uint32_t a = F[i], b = F[l];
                if ((a > b) == ((i & k2) == 0)) { F[i] = b; F[l] = a; }
            }
            __syncwarp();
        }
    }
}

// LSD radix sort of n <= 512 distinct ids (< 2^bits) by one warp in its shared memory: A holds the keys, B is a second buffer
// of the same size, hist 256 words.  Digits of <= 8 bits, counted with shared-memory atomics, scanned (8 bins per lane),
// scattered stably 32 keys at a time (__match_any_sync ranks the keys of equal digit).  Returns the buffer with the result.
// For the list lengths range queries produce (tens to a few hundred) this takes a third of the instructions of the
// bitonic network.
__device__ __forceinline__ uint32_t *pc_warp_radix_sort(uint32_t *A, uint32_t *B, uint32_t *hist, int n, int bits, int lane)
{
    const int passes = (bits + 7) / 8, db = (bits + passes - 1) / passes, bins = 1 << db;
    const uint32_t lt = (1u << lane) - 1u;
    for (int p = 0; p < passes; p++) {
        const int shift = p * db;
        for (int i = lane; i < bins; i += 32) hist[i] = 0u;
        __syncwarp();
        for (int i = lane; i < n; i += 32) atomicAdd(&hist[(A[i] >> shift) & (bins - 1)], 1u);
        __syncwarp();
        {   // exclusive scan of the bins: bins / 32 consecutive ones per lane
            const int per = bins >> 5 ? bins >> 5 : 1, b0 = lane * per;
            uint32_t sum = 0u;
            if (b0 < bins) for (int t = 0; t < per; t++) sum += hist[b0 + t];
            uint32_t incl = sum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(PC_FULL_MASK, incl, d); if (lane >= d) incl += v; }
            uint32_t run = incl - sum;
            if (b0 < bins) for (int t = 0; t < per; t++) { const uint32_t c = hist[b0 + t]; hist[b0 + t] = run; run += c; }
        }
        __syncwarp();
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            const bool valid = i < n;
            const uint32_t key = valid ? A[i] : 0u;
            const uint32_t d = valid ? (key >> shift) & (uint32_t)(bins - 1) : 0x10000u | (uint32_t)lane;      // idle lanes match nobody
            const uint32_t peers = __match_any_sync(PC_FULL_MASK, d);
            const uint32_t rank = __popc(peers & lt);
            uint32_t pos = 0u;
            if (valid) pos = hist[d] + rank;
            __syncwarp();
            if (valid && rank == 0u) hist[d] += __popc(peers);
            if (valid) B[pos] = key;
            __syncwarp();
        }
        uint32_t *t = A; A = B; B = t;
    }
    return A;
}

// ---- the range walk, shared by pc_range_coop_kernel and pc_range_sorted_kernel (range_sorted_kernels.cuh) ----------------
// Query k of a range batch: its point (and in fp64), r2 = range^2 (the inclusive bound of the fp64 test) and the fp32 filter
// thr.  False for an empty index or a NaN range: the query has no hits.
struct pc_range_q {
    float qx, qy, qz;
    double qxd, qyd, qzd;
    double r2;
    float thr;
};

__device__ __forceinline__ bool pc_range_query(const pc_tree &T, const float *__restrict__ q, int64_t k, int qstride,
                                               const double *__restrict__ range, int range_is_scalar, pc_range_q &Q)
{
    const float *qq = q + k * qstride;
    Q.qx = qq[0]; Q.qy = qq[1]; Q.qz = qq[2];
    Q.qxd = (double)Q.qx; Q.qyd = (double)Q.qy; Q.qzd = (double)Q.qz;
    const double r = range[range_is_scalar ? 0 : k];
    Q.r2 = __dmul_rn(r, r);
    if (T.n_points == 0 || !(Q.r2 == Q.r2)) return false;
    Q.thr = fminf(__fmul_ru(__double2float_ru(Q.r2), PC_THR_SLACK), FLT_MAX);
    return true;
}

// One warp walks the tree for one query and returns its number of hits.  The open inner nodes sit on a LIFO frontier of FCAP
// words in F; every step each lane takes one of them and tests its two child boxes; a child that is a leaf is scanned on the
// spot (only its own `count` points: its neighbours' points belong to other leaves), inner children are pushed.  Every
// scanned candidate goes to the sink S, in walk order, as pc_range_hit(S, hit, at, pos, id): `hit` whether it passed the
// test, at() its place in the list, `pos` the point's position in the tree's point array, `id` its original index.  at()
// is a callable so that each sink evaluates it where it needs it: inside or before its `hit` branch.  That choice shapes
// the compiled walk, and each sink keeps the one its kernel was tuned with.  F is free again when the walk returns.
template <int FCAP, class SINK>
__device__ __forceinline__ int64_t pc_range_walk(const pc_tree &T, const pc_range_q &Q, uint32_t *F, int lane, SINK &S)
{
    const float qx = Q.qx, qy = Q.qy, qz = Q.qz, thr = Q.thr;
    const double qxd = Q.qxd, qyd = Q.qyd, qzd = Q.qzd, r2 = Q.r2;
    const uint32_t lt = (1u << lane) - 1u;
    int64_t total = 0;
    int size = 0;
    {
        // start from the seeds (pc_tree_seed_kernel): the leaves met while the top of the tree was expanded -- one per lane, only
        // their own `count` points -- and up to 32 inner nodes for the frontier
        const int n_seed = (int)T.seeds[0], n_seed_leaf = (int)T.seeds[1];
        bool hit[PC_LEAF];
        int32_t id[PC_LEAF];
        uint32_t at0 = 0;
#pragma unroll
        for (int i = 0; i < PC_LEAF; i++) { hit[i] = false; id[i] = 0; }
        if (lane < n_seed_leaf) {
            const uint32_t ref = T.seeds[PC_SEED_LEAF + 2 * lane], cnt = T.seeds[PC_SEED_LEAF + 2 * lane + 1];
            at0 = ref & ~PC_REF_LEAF;
            const float4 *pts = T.points + at0;
#pragma unroll
            for (int i = 0; i < PC_LEAF; i++) {
                if ((uint32_t)i < cnt) {
                    const float4 p = __ldg(pts + i);
                    const float dx = p.x - qx, dy = p.y - qy, dz = p.z - qz;
                    if (fmaf(dz, dz, fmaf(dy, dy, dx * dx)) <= thr) hit[i] = pc_exact_d2(p.x, p.y, p.z, qxd, qyd, qzd) <= r2;
                    id[i] = __float_as_int(p.w);
                }
            }
        }
        if (n_seed_leaf > 0) {
#pragma unroll
            for (int i = 0; i < PC_LEAF; i++) {
                const uint32_t mask = __ballot_sync(PC_FULL_MASK, hit[i]);
                pc_range_hit(S, hit[i], [&] { return total + __popc(mask & lt); }, at0 + i, (uint32_t)id[i]);
                total += __popc(mask);
            }
        }
        if (lane < n_seed) F[lane] = T.seeds[PC_SEED_INNER + lane];
        size = n_seed;
    }
    __syncwarp();
    while (size > 0) {
        // every lane takes one node and pushes at most two; close to the capacity: one node per step (depth-first, at most
        // one more entry per tree level)
        const int take = (size + 64 + PC_STACK <= FCAP) ? min(size, 32) : 1;
        const bool active = lane < take;
        uint32_t node = 0;
        if (active) node = F[size - 1 - lane];
        size -= take;
        __syncwarp();
        bool push0 = false, push1 = false, leaf0 = false, leaf1 = false;
        uint32_t r0 = 0, r1 = 0, c0 = 0, c1 = 0;
        if (active) {
            const pc_rec rec = pc_load_rec(T.rec + 4ull * node);
            const float2 dd = pc_rec_d2(rec, qx, qy, qz);
            const bool in0 = dd.x <= thr, in1 = dd.y <= thr;
            r0 = pc_rec_ref(rec, 0); r1 = pc_rec_ref(rec, 1);
            c0 = pc_rec_cnt(rec, 0); c1 = pc_rec_cnt(rec, 1);
            leaf0 = in0 && (r0 & PC_REF_LEAF); leaf1 = in1 && (r1 & PC_REF_LEAF);
            push0 = in0 && !(r0 & PC_REF_LEAF); push1 = in1 && !(r1 & PC_REF_LEAF);
        }
        if (__ballot_sync(PC_FULL_MASK, leaf0 || leaf1)) {
            bool hit[2 * PC_LEAF];
            int32_t id[2 * PC_LEAF];
#pragma unroll
            for (int c = 0; c < 2; c++) {
                const bool leaf = c ? leaf1 : leaf0;
                const uint32_t cnt = leaf ? (c ? c1 : c0) : 0u;
                const float4 *pts = T.points + ((c ? r1 : r0) & ~PC_REF_LEAF);
#pragma unroll
                for (int i = 0; i < PC_LEAF; i++) {
                    hit[c * PC_LEAF + i] = false; id[c * PC_LEAF + i] = 0;
                    if ((uint32_t)i < cnt) {
                        const float4 p = __ldg(pts + i);
                        const float dx = p.x - qx, dy = p.y - qy, dz = p.z - qz;
                        const float d = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
                        if (d <= thr) hit[c * PC_LEAF + i] = pc_exact_d2(p.x, p.y, p.z, qxd, qyd, qzd) <= r2;
                        id[c * PC_LEAF + i] = __float_as_int(p.w);
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < 2 * PC_LEAF; i++) {
                const uint32_t mask = __ballot_sync(PC_FULL_MASK, hit[i]);
                const uint32_t pos = ((i < PC_LEAF ? r0 : r1) & ~PC_REF_LEAF) + (i % PC_LEAF);
                pc_range_hit(S, hit[i], [&] { return total + __popc(mask & lt); }, pos, (uint32_t)id[i]);
                total += __popc(mask);
            }
        }
        const uint32_t m0 = __ballot_sync(PC_FULL_MASK, push0), m1 = __ballot_sync(PC_FULL_MASK, push1);
        const int n0 = __popc(m0);
        if (push0) F[size + __popc(m0 & lt)] = r0;
        if (push1) F[size + n0 + __popc(m1 & lt)] = r1;
        size += n0 + __popc(m1);
        __syncwarp();
    }
    return total;
}

struct pc_range_stage {                // PC_RANGE_CAPTURE: where the counting pass parks the short lists
    int32_t *stage;                    // stage_cap entries
    unsigned long long stage_cap;
    unsigned long long *cursor;        // next free entry
    int64_t *pos;                      // per query: start of its parked list, -1 = not parked (walk it again)
};

// where pc_range_coop_kernel<MODE> puts a hit's original index: nowhere (COUNT), into its CSR row (FILL), into the warp's
// hit buffer while the list is short enough to be captured (CAPTURE)
template <int MODE>
struct pc_range_sink {
    int32_t *out_idx;
    int64_t begin;
    uint32_t *H;
};

template <int MODE, class AT>
__device__ __forceinline__ void pc_range_hit(pc_range_sink<MODE> &S, bool hit, AT at, uint32_t, uint32_t id)
{
    if (MODE == PC_RANGE_FILL && hit) S.out_idx[S.begin + at()] = (int32_t)id;
    if (MODE == PC_RANGE_CAPTURE && hit) { const int64_t a = at(); if (a < PC_RCAP_HITS) S.H[a] = id; }
}

#define PC_RCAP_FRONT 768         // frontier entries of the capturing pass: 512 double as the sort's second buffer, 256 as its histogram
template <int MODE>
__global__ void __launch_bounds__(32 * PC_RCOOP_WARPS, MODE == PC_RANGE_CAPTURE ? PC_RCAP_MIN_CTAS : (MODE == PC_RANGE_COUNT ? 12 : 8))
pc_range_coop_kernel(pc_tree T, const float *__restrict__ q, int64_t m, int qstride,
                     const double *__restrict__ range, int range_is_scalar,
                     int64_t *__restrict__ counts, const int64_t *__restrict__ offsets, int32_t *__restrict__ out_idx,
                     unsigned long long *__restrict__ long_count, int64_t *__restrict__ long_list,
                     pc_range_stage S, const int64_t *__restrict__ qlist, const unsigned long long *__restrict__ qlist_count)
{
    constexpr bool FILL = MODE == PC_RANGE_FILL;
    constexpr bool CAPTURE = MODE == PC_RANGE_CAPTURE;
    constexpr int FCAP = CAPTURE ? PC_RCAP_FRONT : PC_RCOOP_CAP;
    __shared__ uint32_t s_front[PC_RCOOP_WARPS][FCAP];
    __shared__ uint32_t s_hits[CAPTURE ? PC_RCOOP_WARPS : 1][CAPTURE ? PC_RCAP_HITS : 1];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int64_t k = (int64_t)blockIdx.x * PC_RCOOP_WARPS + w;
    if (qlist) {                       // fill pass over the queries the capture left behind
        if ((unsigned long long)k >= *qlist_count) return;
        k = qlist[k];
    }
    if (k >= m) return;
    uint32_t *H = s_hits[CAPTURE ? w : 0];
    int64_t begin = 0, want = 0;
    if (FILL) {
        begin = offsets[k]; want = offsets[k + 1] - begin;
        if (want == 0) return;
    }
    pc_range_q Q;
    if (!pc_range_query(T, q, k, qstride, range, range_is_scalar, Q)) {
        if (!FILL && lane == 0) counts[k] = 0;
        return;
    }
    uint32_t *F = s_front[w];
    pc_range_sink<MODE> sink = { out_idx, begin, H };
    const int64_t total = pc_range_walk<FCAP>(T, Q, F, lane, sink);
    if (!FILL) {
        if (lane == 0) counts[k] = total;
        if (CAPTURE) {
            // a short list: canonical order (ascending original index) here, then parked until its CSR position is known
            long long start = -1;
            if (total > 0 && total <= PC_RCAP_HITS) {
                __syncwarp();
                // the walk is over: its frontier buffer is free -- second key buffer and the digit histogram
                const int bits = 64 - __clzll((unsigned long long)(T.n_points > 1 ? T.n_points - 1 : 1));
                const uint32_t *sorted = pc_warp_radix_sort(H, F, F + PC_RCAP_HITS, (int)total, bits, lane);
                if (lane == 0) {
                    const unsigned long long at = atomicAdd(S.cursor, (unsigned long long)total);
                    start = at + (unsigned long long)total <= S.stage_cap ? (long long)at : -1;
                }
                start = __shfl_sync(PC_FULL_MASK, start, 0);
                if (start >= 0) for (int i = lane; i < total; i += 32) S.stage[start + i] = (int32_t)sorted[i];
            }
            if (lane == 0) S.pos[k] = start;
        }
        return;
    }
    // canonical order: ascending original index
    if (want <= PC_RFILL_WARP_SORT) {
        int N = 32;
        while (N < want) N <<= 1;
        __syncwarp();
        for (int i = lane; i < N; i += 32) F[i] = i < want ? (uint32_t)out_idx[begin + i] : 0x7fffffffu;
        __syncwarp();
        pc_warp_bitonic(F, N, lane);
        for (int i = lane; i < want; i += 32) out_idx[begin + i] = (int32_t)F[i];
    } else if (lane == 0) {
        long_list[atomicAdd(long_count, 1ull)] = k;            // sorted by pc_range_sort_long_kernel
    }
}

// after the scan: every parked list moves to its CSR position (one warp per query, coalesced); the queries whose lists were
// too long to park are queued for the fill pass
#define PC_RPLACE_WARPS 8
__global__ void __launch_bounds__(32 * PC_RPLACE_WARPS)
pc_range_place_kernel(int64_t m, const int64_t *__restrict__ offsets, const int32_t *__restrict__ stage, const int64_t *__restrict__ pos,
                      int32_t *__restrict__ out_idx, unsigned long long *__restrict__ todo_count, int64_t *__restrict__ todo_list)
{
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * PC_RPLACE_WARPS + (threadIdx.x >> 5);
    if (k >= m) return;
    const int64_t begin = offsets[k], n = offsets[k + 1] - begin;
    if (n == 0) return;
    const int64_t p = pos[k];
    if (p < 0) {
        if (lane == 0) todo_list[atomicAdd(todo_count, 1ull)] = k;
        return;
    }
    for (int64_t i = lane; i < n; i += 32) out_idx[begin + i] = stage[p + i];
}

// lists the fill pass could not sort inside a warp's shared memory: one CTA per queued list, bitonic network over up to
// PC_RLONG_CAP ids in (dynamic) shared memory
#define PC_RLONG_CAP 32768
#define PC_RLONG_THREADS 1024

__global__ void __launch_bounds__(PC_RLONG_THREADS)
pc_range_sort_long_kernel(const unsigned long long *__restrict__ long_count, const int64_t *__restrict__ long_list,
                          const int64_t *__restrict__ offsets, int32_t *__restrict__ out_idx)
{
    extern __shared__ uint32_t s_ids[];
    const unsigned long long n_long = *long_count;
    for (unsigned long long li = blockIdx.x; li < n_long; li += gridDim.x) {
        const int64_t k = long_list[li];
        const int64_t begin = offsets[k], want = offsets[k + 1] - begin;
        if (want > PC_RLONG_CAP) {
            if (threadIdx.x == 0) pc_sort_list(out_idx + begin, want);
            continue;
        }
        int N = 512;
        while (N < want) N <<= 1;
        for (int i = threadIdx.x; i < N; i += PC_RLONG_THREADS) s_ids[i] = i < want ? (uint32_t)out_idx[begin + i] : 0x7fffffffu;
        __syncthreads();
        for (int k2 = 2; k2 <= N; k2 <<= 1) {
            for (int j = k2 >> 1; j > 0; j >>= 1) {
                for (int t = threadIdx.x; t < (N >> 1); t += PC_RLONG_THREADS) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), l = i | j;
                    const uint32_t a = s_ids[i], b = s_ids[l];
                    if ((a > b) == ((i & k2) == 0)) { s_ids[i] = b; s_ids[l] = a; }
                }
                __syncthreads();
            }
        }
        for (int i = threadIdx.x; i < want; i += PC_RLONG_THREADS) out_idx[begin + i] = (int32_t)s_ids[i];
        __syncthreads();
    }
}

// ---- exclusive scan of int64 counts into offsets[m + 1] (three small kernels) ---------------------------
#define PC_SCAN_THREADS 256
#define PC_SCAN_ITEMS 8
#define PC_SCAN_TILE (PC_SCAN_THREADS * PC_SCAN_ITEMS)

__device__ __forceinline__ int64_t pc_block_exclusive_scan(int64_t v, int64_t *total)
{
    __shared__ int64_t warp_sum[PC_SCAN_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int64_t t = __shfl_up_sync(PC_FULL_MASK, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    int64_t woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < PC_SCAN_THREADS / 32; w++) { if (w < warp) woff += warp_sum[w]; tot += warp_sum[w]; }
    if (total) *total = tot;
    return woff + incl - v;
}

__global__ void __launch_bounds__(PC_SCAN_THREADS)
pc_scan_tile_sums(const int64_t *__restrict__ counts, int64_t m, int64_t *__restrict__ tile_sum)
{
    const int64_t base = (int64_t)blockIdx.x * PC_SCAN_TILE + (int64_t)threadIdx.x * PC_SCAN_ITEMS;
    int64_t s = 0;
#pragma unroll
    for (int i = 0; i < PC_SCAN_ITEMS; i++) if (base + i < m) s += counts[base + i];
    int64_t tot;
    pc_block_exclusive_scan(s, &tot);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(PC_SCAN_THREADS)
pc_scan_tile_offsets(int64_t *__restrict__ tile_sum, int64_t n_tiles)
{
    __shared__ int64_t carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int64_t base = 0; base < n_tiles; base += PC_SCAN_THREADS) {
        int64_t i = base + threadIdx.x;
        int64_t v = i < n_tiles ? tile_sum[i] : 0, tot;
        int64_t ex = pc_block_exclusive_scan(v, &tot);
        int64_t carry = carry_s;
        if (i < n_tiles) tile_sum[i] = carry + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + tot;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(PC_SCAN_THREADS)
pc_scan_write_offsets(const int64_t *__restrict__ counts, int64_t m, const int64_t *__restrict__ tile_off,
                      int64_t *__restrict__ offsets)
{
    const int64_t base = (int64_t)blockIdx.x * PC_SCAN_TILE + (int64_t)threadIdx.x * PC_SCAN_ITEMS;
    int64_t c[PC_SCAN_ITEMS], s = 0;
#pragma unroll
    for (int i = 0; i < PC_SCAN_ITEMS; i++) { c[i] = base + i < m ? counts[base + i] : 0; s += c[i]; }
    int64_t run = tile_off[blockIdx.x] + pc_block_exclusive_scan(s, nullptr);
#pragma unroll
    for (int i = 0; i < PC_SCAN_ITEMS; i++) {
        if (base + i < m) offsets[base + i] = run;
        run += c[i];
        if (base + i == m - 1) offsets[m] = run;
    }
}

// ---- sensing gather: every point within `radius` of one centre ---------------------------------------------------
// The LiDAR-mode sensor of the reference gathers the observed map with ONE radius search of ~20 m on the global cloud
// (Planner/src/camera_sensor.cpp:133-145).  A result of 10^5..10^6 points is a stream compaction, not a tree walk:
// every point is tested (fp32 filter, fp64 decision as everywhere), hits are appended CTA by CTA, and the list is then
// radix-sorted by original index.
__global__ void __launch_bounds__(256)
pc_sphere_gather_kernel(const float4 *__restrict__ points, int64_t n, float cx, float cy, float cz, double r2, float thr,
                        uint32_t *__restrict__ out, unsigned long long cap, unsigned long long *__restrict__ count)
{
    __shared__ uint32_t s_warp[8];
    __shared__ unsigned long long s_base;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    bool hit = false;
    uint32_t id = 0;
    if (i < n) {
        const float4 p = __ldg(points + i);
        const float dx = p.x - cx, dy = p.y - cy, dz = p.z - cz;
        const float d = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
        if (d <= thr) hit = pc_exact_d2(p.x, p.y, p.z, (double)cx, (double)cy, (double)cz) <= r2;
        id = __float_as_uint(p.w);
    }
    const uint32_t mask = __ballot_sync(PC_FULL_MASK, hit);
    if (lane == 0) s_warp[warp] = __popc(mask);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int w = 0; w < 8; w++) { const uint32_t c = s_warp[w]; s_warp[w] = tot; tot += c; }
        s_base = tot ? atomicAdd(count, (unsigned long long)tot) : 0ull;
    }
    __syncthreads();
    if (hit) {
        const unsigned long long pos = s_base + s_warp[warp] + __popc(mask & pc_lanemask_lt());
        if (pos < cap) out[pos] = id;
    }
}
