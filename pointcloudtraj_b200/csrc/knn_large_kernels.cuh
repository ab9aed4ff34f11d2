// knn_large_kernels.cuh -- pc_knn_large_batch: exact k-nearest-neighbour rows for PC_KNN_MAX < k <= PC_KNN_LARGE_MAX.
//
// Same rows as pc_knn_batch (knn_kernels.cuh): the k smallest (fp64 d2 = pc_exact_d2, original index), the optional bound
// d2 <= r2, padding (-1, +inf).  The walk is pc_knn_warp_search, one WARP per query (seeds, then up to 32 frontier nodes a
// step, fp32 box / point filter against thr, the fp64 re-check of every survivor, leaves over their own counts).  Only the
// list differs: a k-list spread over the lanes holds at most 32 entries, so here it lives in shared memory:
//   list   the first n (<= k) entries, ascending by (d2, index): 12 k bytes per warp
//   queue  PC_KNNL_QUEUE candidates that passed the re-check, the bound and the k-th entry when they were offered, appended
//          by ballot prefix.  thr is only refreshed by a flush, so it may lag behind the queue: that costs filter work, not
//          correctness, since every queued entry is ranked again by the merge.
//   flush  (when the next offer could overflow the queue, and at the end of the walk) a warp bitonic sort of the queue under
//          the exact (d2, index) order, then a merge by rank: an entry's new position is its own position plus the number of
//          entries of the other sequence before it (binary search).  (d2, index) pairs are distinct -- a point is scanned once
//          per query -- so the map is strictly increasing and list entries only move up: the merge runs in place, in chunks
//          of 32 from the top, and drops every position >= k.
#pragma once
#include "knn_kernels.cuh"
#include "range_sorted_kernels.cuh"     // pc_pair_bitonic

#define PC_KNN_LARGE_WARPS 2            // warps per CTA: 42.5 KB of dynamic shared memory at k = 1024, 5 CTAs per SM
#define PC_KNNL_QUEUE 64                // candidate queue per warp (entries)

// dynamic shared memory of one warp: the frontier (uint2), the queue's and the list's d2, then their indices
__host__ __device__ __forceinline__ size_t pc_knnl_warp_bytes(int k)
{
    const size_t b = (size_t)PC_KNN_FRONT * sizeof(uint2) + (size_t)(PC_KNNL_QUEUE + k) * (sizeof(double) + sizeof(uint32_t));
    return (b + 15) & ~(size_t)15;      // the next warp's doubles stay aligned for odd k
}

struct pc_knn_qlist {
    double *QD;                         // queue: PC_KNNL_QUEUE entries, the first qn used, unordered
    double *D;                          // list: k entries, the first n valid
    uint32_t *QI, *I;
    int n, qn;                          // warp-uniform
    double kd;                          // the k-th entry (+inf, PC_KNN_NONE while n < k); thr as in pc_knn_wlist
    uint32_t ki;
    float thr;
};

// number of the first len entries of (D, I) that come before (e, id) in the row order
__device__ __forceinline__ int pc_knnl_rank(const double *D, const uint32_t *I, int len, double e, uint32_t id)
{
    int lo = 0, hi = len;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (pc_knn_less(D[mid], I[mid], e, id)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Sort the queue (qn > 0 entries), merge it into the list (n entries), return the list's new length.  Called by the whole
// warp; kept out of line (one copy for the many offer sites of the unrolled scans) with scalar arguments only.
__device__ __noinline__ int pc_knnl_flush(int lane, int k, int n, int qn, double *QD, uint32_t *QI, double *D, uint32_t *I)
{
    __syncwarp();
    pc_pair_bitonic<32, int>(QD, QI, qn, lane);
    // the queue's new positions, from the old list (held in registers while the list moves)
    double qe[PC_KNNL_QUEUE / 32];
    uint32_t qi[PC_KNNL_QUEUE / 32];
    int qpos[PC_KNNL_QUEUE / 32];
#pragma unroll
    for (int c = 0; c < PC_KNNL_QUEUE / 32; c++) {
        const int j = lane + 32 * c;
        qe[c] = 0.0; qi[c] = 0u; qpos[c] = k;
        if (j < qn) {
            qe[c] = QD[j]; qi[c] = QI[j];
            qpos[c] = j + pc_knnl_rank(D, I, n, qe[c], qi[c]);
        }
    }
    // list entries before the smallest queued one stay; from there on entry i moves to i + (queued entries before it), and
    // entries at k - 1 and above are pushed out
    const int p0 = __shfl_sync(PC_FULL_MASK, qpos[0], 0);
    for (int hi = min(n, k - 1); hi > p0; hi -= 32) {
        const int i = hi - 1 - lane;
        double e = 0.0;
        uint32_t id = 0u;
        int to = k;
        if (i >= p0) { e = D[i]; id = I[i]; to = i + pc_knnl_rank(QD, QI, qn, e, id); }
        __syncwarp();
        if (to < k) { D[to] = e; I[to] = id; }
        __syncwarp();
    }
#pragma unroll
    for (int c = 0; c < PC_KNNL_QUEUE / 32; c++)
        if (qpos[c] < k) { D[qpos[c]] = qe[c]; I[qpos[c]] = qi[c]; }
    __syncwarp();
    return min(k, n + qn);
}

__device__ __forceinline__ void pc_knnl_flush(int lane, const pc_knn_dev &K, pc_knn_qlist &W)
{
    W.n = pc_knnl_flush(lane, K.k, W.n, W.qn, W.QD, W.QI, W.D, W.I);
    W.qn = 0;
    if (W.n == K.k) { W.kd = W.D[K.k - 1]; W.ki = W.I[K.k - 1]; }
    W.thr = fminf(K.bound_thr, pc_thr_from(W.kd));
}

// the pc_knn_warp_scan offer of pc_knn_qlist: every lane's candidate that still comes before the k-th entry is queued
__device__ __forceinline__ void pc_knn_warp_insert(bool have, double e, uint32_t id, int lane, const pc_knn_dev &K, pc_knn_qlist &W)
{
    const uint32_t lt = (1u << lane) - 1u;
    have = have && pc_knn_less(e, id, W.kd, W.ki);
    uint32_t b = __ballot_sync(PC_FULL_MASK, have);
    if (b == 0u) return;
    if (W.qn + __popc(b) > PC_KNNL_QUEUE) {
        pc_knnl_flush(lane, K, W);
        have = have && pc_knn_less(e, id, W.kd, W.ki);
        b = __ballot_sync(PC_FULL_MASK, have);
    }
    if (have) { const int at = W.qn + __popc(b & lt); W.QD[at] = e; W.QI[at] = id; }
    W.qn += __popc(b);
}

// One warp per query: slot t of the batch (perm / ordered: the curve order of the ordering pass, m_eff its query count)
__global__ void __launch_bounds__(32 * PC_KNN_LARGE_WARPS)
pc_knn_large_kernel(pc_tree T, pc_knn_dev K, const float *__restrict__ q, int64_t m, int qstride,
                    const uint32_t *__restrict__ perm, const float4 *__restrict__ ordered, const unsigned long long *__restrict__ m_eff,
                    int32_t *__restrict__ out_idx, float *__restrict__ out_d2)
{
    extern __shared__ __align__(16) unsigned char s_knnl[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned char *base = s_knnl + (size_t)w * pc_knnl_warp_bytes(K.k);
    uint2 *F = reinterpret_cast<uint2 *>(base);
    pc_knn_qlist W;
    W.QD = reinterpret_cast<double *>(base + (size_t)PC_KNN_FRONT * sizeof(uint2));
    W.D = W.QD + PC_KNNL_QUEUE;
    W.QI = reinterpret_cast<uint32_t *>(W.D + K.k);
    W.I = W.QI + PC_KNNL_QUEUE;
    const long long m_search = m_eff ? (long long)*m_eff : (long long)m;
    const long long n_warps = (long long)gridDim.x * PC_KNN_LARGE_WARPS;
    for (long long t = (long long)blockIdx.x * PC_KNN_LARGE_WARPS + w; t < m_search; t += n_warps) {
        uint32_t slot;
        float qx, qy, qz;
        pc_knn_fetch(q, qstride, perm, ordered, t, slot, qx, qy, qz);
        W.n = W.qn = 0;
        W.kd = INFINITY; W.ki = PC_KNN_NONE; W.thr = K.bound_thr;
        if (T.n_points > 0) pc_knn_warp_search(T, K, qx, qy, qz, F, lane, W);
        if (W.qn > 0) pc_knnl_flush(lane, K, W);
        const size_t o = (size_t)slot * K.k;
        for (int j = lane; j < K.k; j += 32) {
            const bool real = j < W.n;
            if (out_idx) out_idx[o + j] = real ? (int32_t)W.I[j] : -1;
            if (out_d2) out_d2[o + j] = real ? (float)W.D[j] : INFINITY;
        }
        __syncwarp();
    }
}
