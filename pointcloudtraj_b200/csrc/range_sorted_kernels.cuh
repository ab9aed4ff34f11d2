// range_sorted_kernels.cuh -- pc_range_sorted_batch: the hit lists of range queries ordered by (fp64 d2, original index) and
// cut to max_nn (pcl::search::KdTree::radiusSearch with k_sqr_distances and max_nn).
//
// The hit set is pc_range_batch's (range_kernels.cuh): the same walk (pc_range_walk), fp32 filter and inclusive fp64 test.  What differs is
// what a hit is remembered by and how a list is sorted:
//   - the walk records a hit by its POSITION in the tree's point array (4 bytes).  After the walk the warp reads the point
//     again (L1 / L2), recomputes its fp64 d2 with pc_exact_d2 -- the value the hit test used -- and its original index;
//   - a list is sorted by (fp64 d2, index) with a bitonic network over (double, uint32) pairs, compared exactly: no key
//     compression, no fix-up pass.
// One WARP per query.  The capturing pass sorts lists of up to PC_RS_CAP_HITS hits in the warp's shared memory: the 1024-word
// frontier, free once the walk is over, holds their 512 fp64 d2, the hit buffer their indices.  The first max_nn entries are
// parked as (index, float32 d2) pairs until the scan of the truncated counts gives their CSR position.  Longer lists are queued
// with their untruncated length, walked a second time into a scratch area (fill pass) and sorted by one CTA each, in shared
// memory up to PC_RS_LONG_CAP entries and in the scratch area (global memory) beyond.
#pragma once
#include "range_kernels.cuh"

#define PC_RS_WARPS 4
#define PC_RS_CAP_HITS 512         // lists sorted by the capturing warp
#define PC_RS_FRONT 1024           // frontier words per warp: after the walk, the PC_RS_CAP_HITS doubles of the sort
#ifndef PC_RS_MIN_CTAS
#define PC_RS_MIN_CTAS 8           // 24 KB of shared memory per CTA: 8 CTAs fit an SM
#endif
#define PC_RS_LONG_CAP 16384       // pairs a CTA sorts in (dynamic) shared memory: 192 KB
#define PC_RS_LONG_THREADS 1024
#define PC_RS_CAPTURE 0
#define PC_RS_FILL 1

struct pc_rs_args {
    int64_t *counts;                   // capture: per query min(hits, max_nn)
    int32_t *stage_idx;                // capture: parked lists, (index, float32 d2), stage_cap entries
    float *stage_d2;
    unsigned long long stage_cap;
    unsigned long long *cursor;        // [0] next free stage entry, [1] long lists, [2] scratch entries of the long lists
    int64_t *pos;                      // per query: start of its parked list, -1 = a long list
    int64_t *long_list;                // per long list: query, scratch start, untruncated length
    double *long_d2;                   // fill: the long lists in the scratch area (fp64 d2, original index)
    uint32_t *long_ref;
};

// ascending compare-exchange under (d2, index)
template <typename IT>
__device__ __forceinline__ void pc_pair_cx(double *D, uint32_t *I, IT i, IT l)
{
    const double a = D[i], b = D[l];
    const uint32_t x = I[i], y = I[l];
    if (a > b || (a == b && x > y)) { D[i] = b; D[l] = a; I[i] = y; I[l] = x; }
}

// bitonic sort of n (d2, index) pairs, ascending, by NT threads (this one is `tid`).  The network is that of the next power of
// two, in the form where every compare-exchange puts the smaller key at the lower position (each merge starts by comparing
// mirrored entries): the entries past n count as +inf, never move, and need no storage.
template <int NT, typename IT>
__device__ __forceinline__ void pc_pair_bitonic(double *D, uint32_t *I, IT n, int tid)
{
    IT N = 1;
    while (N < n) N <<= 1;
    for (IT k2 = 2; k2 <= N; k2 <<= 1) {
        for (IT j = k2 >> 1; j > 0; j >>= 1) {
            for (IT t = tid; t < (N >> 1); t += NT) {
                const IT i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const IT l = j == (k2 >> 1) ? i ^ (k2 - 1) : i | j;
                if (l < n) pc_pair_cx<IT>(D, I, i, l);
            }
            if (NT == 32) __syncwarp(); else __syncthreads();
        }
    }
}

// where pc_range_sorted_kernel<MODE> puts a hit's tree position: into the scratch area of its long list (FILL), into the warp's
// hit buffer while the list is short enough to be captured (CAPTURE)
template <int MODE>
struct pc_rs_sink {
    uint32_t *out;
    uint32_t *H;
};

template <int MODE, class AT>
__device__ __forceinline__ void pc_range_hit(pc_rs_sink<MODE> &S, bool hit, AT at, uint32_t pos, uint32_t)
{
    if (MODE == PC_RS_FILL && hit) S.out[at()] = pos;
    if (MODE == PC_RS_CAPTURE) { const int64_t a = at(); if (hit && a < PC_RS_CAP_HITS) S.H[a] = pos; }
}

// one warp per query: pc_range_walk, recording hit positions
template <int MODE>
__global__ void __launch_bounds__(32 * PC_RS_WARPS, MODE == PC_RS_CAPTURE ? PC_RS_MIN_CTAS : 8)
pc_range_sorted_kernel(pc_tree T, const float *__restrict__ q, int64_t m, int qstride, const double *__restrict__ range,
                       int range_is_scalar, int64_t max_nn, pc_rs_args A, int64_t n_long)
{
    constexpr bool FILL = MODE == PC_RS_FILL;
    constexpr bool CAPTURE = MODE == PC_RS_CAPTURE;
    __shared__ __align__(16) uint32_t s_front[PC_RS_WARPS][PC_RS_FRONT];
    __shared__ uint32_t s_hits[CAPTURE ? PC_RS_WARPS : 1][CAPTURE ? PC_RS_CAP_HITS : 1];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int64_t k = (int64_t)blockIdx.x * PC_RS_WARPS + w, base = 0;
    if (FILL) {
        if (k >= n_long) return;
        base = A.long_list[3 * k + 1];
        k = A.long_list[3 * k];
    }
    if (k >= m) return;
    uint32_t *H = s_hits[CAPTURE ? w : 0];
    uint32_t *out = A.long_ref + base;
    pc_range_q Q;
    if (!pc_range_query(T, q, k, qstride, range, range_is_scalar, Q)) {
        if (CAPTURE && lane == 0) A.counts[k] = 0;
        return;
    }
    uint32_t *F = s_front[w];
    pc_rs_sink<MODE> sink = { out, H };
    const int64_t total = pc_range_walk<PC_RS_FRONT>(T, Q, F, lane, sink);
    __syncwarp();
    if (FILL) {
        // positions -> (fp64 d2, original index), in place; the CTA sort (pc_range_sorted_long_kernel) takes it from here
        for (int64_t i = lane; i < total; i += 32) {
            const float4 p = __ldg(T.points + out[i]);
            A.long_d2[base + i] = pc_exact_d2(p.x, p.y, p.z, Q.qxd, Q.qyd, Q.qzd);
            out[i] = __float_as_uint(p.w);
        }
        return;
    }
    const int64_t keep = max_nn > 0 && max_nn < total ? max_nn : total;
    if (lane == 0) A.counts[k] = keep;
    long long start = -1;
    if (total > 0 && total <= PC_RS_CAP_HITS) {
        // the walk is over: its frontier holds the d2, the hit buffer turns from positions into indices
        double *D = reinterpret_cast<double *>(F);
        for (int i = lane; i < (int)total; i += 32) {
            const float4 p = __ldg(T.points + H[i]);
            D[i] = pc_exact_d2(p.x, p.y, p.z, Q.qxd, Q.qyd, Q.qzd);
            H[i] = __float_as_uint(p.w);
        }
        __syncwarp();
        pc_pair_bitonic<32, int>(D, H, (int)total, lane);
        if (lane == 0) {
            const unsigned long long at = atomicAdd(A.cursor, (unsigned long long)keep);
            start = at + (unsigned long long)keep <= A.stage_cap ? (long long)at : -1;
        }
        start = __shfl_sync(PC_FULL_MASK, start, 0);
        if (start >= 0) {
            for (int i = lane; i < (int)keep; i += 32) {
                A.stage_idx[start + i] = (int32_t)H[i];
                A.stage_d2[start + i] = __double2float_rn(D[i]);
            }
        }
    }
    if (lane == 0) {
        A.pos[k] = start;
        if (start < 0 && total > 0) {           // walked again by the fill pass, into a scratch area of its full length
            const unsigned long long li = atomicAdd(A.cursor + 1, 1ull);
            A.long_list[3 * li] = k;
            A.long_list[3 * li + 1] = (int64_t)atomicAdd(A.cursor + 2, (unsigned long long)total);
            A.long_list[3 * li + 2] = total;
        }
    }
}

// offsets-only calls count with pc_range_coop_kernel<PC_RANGE_COUNT>; the rows are then cut to max_nn
__global__ void pc_range_clamp_kernel(int64_t *__restrict__ counts, int64_t m, int64_t max_nn)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m && counts[k] > max_nn) counts[k] = max_nn;
}

// after the scan: every parked list moves to its CSR position (one warp per query)
__global__ void __launch_bounds__(32 * PC_RPLACE_WARPS)
pc_range_sorted_place_kernel(int64_t m, const int64_t *__restrict__ offsets, const int32_t *__restrict__ stage_idx,
                             const float *__restrict__ stage_d2, const int64_t *__restrict__ pos,
                             int32_t *__restrict__ out_idx, float *__restrict__ out_d2)
{
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * PC_RPLACE_WARPS + (threadIdx.x >> 5);
    if (k >= m) return;
    const int64_t begin = offsets[k], n = offsets[k + 1] - begin;
    if (n == 0) return;
    const int64_t p = pos[k];
    if (p < 0) return;                   // a long list: pc_range_sorted_long_kernel writes it
    for (int64_t i = lane; i < n; i += 32) {
        out_idx[begin + i] = stage_idx[p + i];
        if (out_d2) out_d2[begin + i] = stage_d2[p + i];
    }
}

// the long lists, one CTA each: sorted in shared memory up to PC_RS_LONG_CAP pairs, in their scratch area beyond; the first
// max_nn entries go to the row
__global__ void __launch_bounds__(PC_RS_LONG_THREADS, 1)
pc_range_sorted_long_kernel(int64_t n_long, const int64_t *__restrict__ long_list, double *long_d2, uint32_t *long_ref,
                            const int64_t *__restrict__ offsets, int32_t *__restrict__ out_idx,
                            float *__restrict__ out_d2)
{
    extern __shared__ double s_d2[];
    uint32_t *s_ref = reinterpret_cast<uint32_t *>(s_d2 + PC_RS_LONG_CAP);
    for (int64_t li = blockIdx.x; li < n_long; li += gridDim.x) {
        const int64_t k = long_list[3 * li], base = long_list[3 * li + 1], n = long_list[3 * li + 2];
        double *D = long_d2 + base;
        uint32_t *I = long_ref + base;
        if (n <= PC_RS_LONG_CAP) {
            for (int i = threadIdx.x; i < (int)n; i += PC_RS_LONG_THREADS) { s_d2[i] = D[i]; s_ref[i] = I[i]; }
            __syncthreads();
            D = s_d2; I = s_ref;
            pc_pair_bitonic<PC_RS_LONG_THREADS, int>(D, I, (int)n, threadIdx.x);
        } else {
            pc_pair_bitonic<PC_RS_LONG_THREADS, int64_t>(D, I, n, threadIdx.x);
        }
        const int64_t begin = offsets[k], keep = offsets[k + 1] - begin;
        for (int64_t i = threadIdx.x; i < keep; i += PC_RS_LONG_THREADS) {
            out_idx[begin + i] = (int32_t)I[i];
            if (out_d2) out_d2[begin + i] = __double2float_rn(D[i]);
        }
        __syncthreads();
    }
}
