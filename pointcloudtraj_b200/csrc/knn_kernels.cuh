// knn_kernels.cuh -- exact k-nearest-neighbour batches (pc_knn_batch), with an optional range bound.
//
// The k smallest points of every query under the order (fp64 d2, original index), d2 = pc_exact_d2 (the reference's
// expression); with a bound r >= 0 only points with d2 <= r2 = __dmul_rn(r, r) are candidates (pc_range_batch's test).
// Rows with fewer than k points are padded with (idx -1, d2 +inf).  Exactness as in query_kernels.cuh: boxes and points are
// filtered in fp32 against thr = min(bound, pc_thr_from(d2 of the current k-th entry)), and EVERY point that passes gets the
// fp64 re-check.  Two rules differ from the 1-NN walks:
//   * a leaf is scanned over its own `cnt` points only -- the 1-NN scans read PC_LEAF points from any start (the points
//     behind a short leaf are real points too, and pad copies of the last one), harmless for a minimum but a duplicate entry
//     in a k-list;
//   * no pc_exact_leaf shortcut: "only points within the leaf minimum's margin" holds for the minimum alone.
//
//   pc_knn_coop_kernel    one WARP per query: the frontier walk of pc_query_coop_kernel, the k-list spread over the warp
//                         (lane j holds the j-th entry); also answers the queries of the packets the packet kernel puts aside
//   pc_knn_packet_kernel  one warp walks the tree once for the 32 neighbouring queries of a curve-ordered batch (the walk of
//                         pc_packet_traverse); every lane keeps its query's k-list in shared memory
// The warp walk (pc_knn_warp_search) is a template over the list, shared with pc_knn_large_kernel (knn_large_kernels.cuh).
#pragma once
#include "query_kernels.cuh"

#define PC_KNN_WARPS 4                  // warps per CTA of both kNN kernels
#define PC_KNN_FRONT 1024               // frontier entries per warp of the coop kernel (8 KB)
#define PC_KNN_NONE 0xffffffffu         // index of a padding entry (-1 as int32)

struct pc_knn_dev {
    int k;                              // entries per row, 1..PC_KNN_MAX
    double r2;                          // bound on the fp64 d2 (inclusive), +inf when unbounded
    float bound_thr;                    // fp32 filter of the bound, FLT_MAX when unbounded
    float packet_split;                 // pc_knn_packet_kernel: Chebyshev extent beyond which a packet is deferred (0 = never)
    unsigned long long *defer_count;    // deferred packets (packet kernel) / deferred mode of the coop kernel (non-null)
    uint32_t *defer_list;
};

// (e, id) before (d, di) in the row order; padding entries (+inf, PC_KNN_NONE) come after every point
__device__ __forceinline__ bool pc_knn_less(double e, uint32_t id, double d, uint32_t di)
{
    return e < d || (e == d && id < di);
}

// query t of a batch: slot t, perm[t] (radix-sorted order) or the gathered float4 of the cell-binned order
__device__ __forceinline__ void pc_knn_fetch(const float *__restrict__ q, int qstride, const uint32_t *__restrict__ perm,
                                             const float4 *__restrict__ ordered, long long t, uint32_t &slot, float &qx, float &qy, float &qz)
{
    if (ordered) { const float4 v = ordered[t]; qx = v.x; qy = v.y; qz = v.z; slot = __float_as_uint(v.w); }
    else { slot = perm ? perm[t] : (uint32_t)t; const float *qq = q + (size_t)slot * qstride; qx = qq[0]; qy = qq[1]; qz = qq[2]; }
}

// ---- one warp per query ------------------------------------------------------------------------------------------------
// The warp's k-list: lane j < k holds entry j (ld, li); every lane holds a copy of the k-th entry (kd, ki) and of thr.
struct pc_knn_wlist {
    double ld, kd;
    uint32_t li, ki;
    float thr;
};

// Offer every lane's candidate (have: passed the fp32 filter, the fp64 re-check and the bound) to the list, one lane at a
// time: rank = number of entries before it (ballot), entries from there on move up one lane.  Called by the whole warp.
__device__ __forceinline__ void pc_knn_warp_insert(bool have, double e, uint32_t id, int lane, const pc_knn_dev &K, pc_knn_wlist &W)
{
    uint32_t pend = __ballot_sync(PC_FULL_MASK, have && pc_knn_less(e, id, W.kd, W.ki));
    while (pend) {
        const int src = __ffs(pend) - 1;
        pend &= pend - 1u;
        const double ce = __shfl_sync(PC_FULL_MASK, e, src);
        const uint32_t ci = __shfl_sync(PC_FULL_MASK, id, src);
        if (!pc_knn_less(ce, ci, W.kd, W.ki)) continue;             // an earlier candidate of this round pushed it out
        const int pos = __popc(__ballot_sync(PC_FULL_MASK, lane < K.k && pc_knn_less(W.ld, W.li, ce, ci)));
        const double up_d = __shfl_up_sync(PC_FULL_MASK, W.ld, 1);
        const uint32_t up_i = __shfl_up_sync(PC_FULL_MASK, W.li, 1);
        if (lane == pos) { W.ld = ce; W.li = ci; }
        else if (lane > pos) { W.ld = up_d; W.li = up_i; }
        W.kd = __shfl_sync(PC_FULL_MASK, W.ld, K.k - 1);
        W.ki = __shfl_sync(PC_FULL_MASK, W.li, K.k - 1);
    }
    W.thr = fminf(K.bound_thr, pc_thr_from(W.kd));
}

// scan NL leaves per lane (ref with PC_REF_LEAF, cnt points each; cnt 0 = none) and offer the survivors to the list.
// LIST: pc_knn_wlist (this file) or pc_knn_qlist (knn_large_kernels.cuh); each has its pc_knn_warp_insert and a warp-uniform
// filter W.thr.
template <int NL, typename LIST>
__device__ __forceinline__ void pc_knn_warp_scan(const pc_tree &T, const uint32_t (&ref)[NL], const uint32_t (&cnt)[NL],
                                                 float qx, float qy, float qz, int lane, const pc_knn_dev &K, LIST &W)
{
    float d[NL * PC_LEAF];
#pragma unroll
    for (int c = 0; c < NL; c++) {
#pragma unroll
        for (int i = 0; i < PC_LEAF; i++) {
            d[c * PC_LEAF + i] = INFINITY;
            if ((uint32_t)i < cnt[c]) {
                const float4 p = __ldg(T.points + (ref[c] & ~PC_REF_LEAF) + i);
                const float dx = p.x - qx, dy = p.y - qy, dz = p.z - qz;
                d[c * PC_LEAF + i] = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
            }
        }
    }
    // the candidates in turn (thr tightens as the list fills); a survivor's point is read again (L1) for the fp64 re-check
#pragma unroll
    for (int j = 0; j < NL * PC_LEAF; j++) {
        bool have = (uint32_t)(j % PC_LEAF) < cnt[j / PC_LEAF] && d[j] <= W.thr;
        double e = 0.0;
        uint32_t id = 0u;
        if (have) {
            const float4 p = __ldg(T.points + (ref[j / PC_LEAF] & ~PC_REF_LEAF) + (j % PC_LEAF));
            e = pc_exact_d2(p.x, p.y, p.z, (double)qx, (double)qy, (double)qz);
            id = (uint32_t)__float_as_int(p.w);
            have = e <= K.r2;
        }
        pc_knn_warp_insert(have, e, id, lane, K, W);
    }
}

template <typename LIST>
__device__ __forceinline__ void pc_knn_warp_search(const pc_tree &T, const pc_knn_dev &K, float qx, float qy, float qz,
                                                   uint2 *__restrict__ F, int lane, LIST &W)
{
    const uint32_t lt = (1u << lane) - 1u;
    // the seeds: leaves met while the top of the tree was expanded (one per lane, their own counts) and <= 32 inner nodes
    const int n_seed = (int)T.seeds[0], n_seed_leaf = (int)T.seeds[1];
    for (int base = 0; base < n_seed_leaf; base += 32) {
        uint32_t ref[1] = { 0u }, cnt[1] = { 0u };
        if (base + lane < n_seed_leaf) { ref[0] = T.seeds[PC_SEED_LEAF + 2 * (base + lane)]; cnt[0] = T.seeds[PC_SEED_LEAF + 2 * (base + lane) + 1]; }
        pc_knn_warp_scan<1>(T, ref, cnt, qx, qy, qz, lane, K, W);
    }
    if (lane < n_seed) F[lane] = make_uint2(T.seeds[PC_SEED_INNER + lane], 0u);
    int size = n_seed;
    __syncwarp();
    while (size > 0) {
        // one node per lane from the top of the frontier; close to the capacity one node per step (depth-first)
        const int take = (size + 32 + PC_STACK <= PC_KNN_FRONT) ? min(size, 32) : 1;
        bool active = lane < take;
        uint2 en = make_uint2(0u, 0u);
        if (active) en = F[size - 1 - lane];
        size -= take;
        __syncwarp();
        active = active && __uint_as_float(en.y) <= W.thr;
        float dn = INFINITY, df = INFINITY;          // inner children to push (INFINITY: none)
        uint32_t cn = 0, cf = 0;
        uint32_t ref[2] = { 0u, 0u }, cnt[2] = { 0u, 0u };   // leaf children to scan
        if (active) {
            const pc_rec rec = pc_load_rec(T.rec + 4ull * en.x);
            const float2 dd = pc_rec_d2(rec, qx, qy, qz);
            const bool first0 = dd.x <= dd.y;
            const uint32_t r0 = pc_rec_ref(rec, 0), r1 = pc_rec_ref(rec, 1);
            const uint32_t rn = first0 ? r0 : r1, rf = first0 ? r1 : r0;
            const uint32_t kn = pc_rec_cnt(rec, first0 ? 0 : 1), kf = pc_rec_cnt(rec, first0 ? 1 : 0);
            const float dnn = fminf(dd.x, dd.y), dff = fmaxf(dd.x, dd.y);
            if (dnn <= W.thr) {
                if (rn & PC_REF_LEAF) { ref[0] = rn; cnt[0] = kn; }
                else { cn = rn; dn = dnn; }
            }
            if (dff <= W.thr) {
                if (rf & PC_REF_LEAF) { ref[1] = rf; cnt[1] = kf; }
                else { cf = rf; df = dff; }
            }
        }
        if (__ballot_sync(PC_FULL_MASK, (cnt[0] | cnt[1]) != 0u)) pc_knn_warp_scan<2>(T, ref, cnt, qx, qy, qz, lane, K, W);
        // push the inner children that survive the (possibly tightened) bound, the nearer ones on top
        const bool wn = dn <= W.thr, wf = df <= W.thr;
        const uint32_t mf = __ballot_sync(PC_FULL_MASK, wf), mn = __ballot_sync(PC_FULL_MASK, wn);
        const int nf = __popc(mf), nn = __popc(mn);
        if (wf) F[size + __popc(mf & lt)] = make_uint2(cf, __float_as_uint(df));
        if (wn) F[size + nf + (nn - 1 - __popc(mn & lt))] = make_uint2(cn, __float_as_uint(dn));
        size += nf + nn;
        __syncwarp();
    }
}

// Work items: the m queries of the batch (K.defer_count == nullptr), or the queries of the packets pc_knn_packet_kernel put
// on K.defer_list (32 per packet, curve-ordered batch: perm / ordered / m_eff as for the packet kernel).
__global__ void __launch_bounds__(32 * PC_KNN_WARPS)
pc_knn_coop_kernel(pc_tree T, pc_knn_dev K, const float *__restrict__ q, int64_t m, int qstride,
                   const uint32_t *__restrict__ perm, const float4 *__restrict__ ordered, const unsigned long long *__restrict__ m_eff,
                   int32_t *__restrict__ out_idx, float *__restrict__ out_d2)
{
    __shared__ uint2 s_front[PC_KNN_WARPS][PC_KNN_FRONT];       // (inner node, float bits of its box distance)
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long m_search = m_eff ? (long long)*m_eff : (long long)m;
    const unsigned long long n_items = K.defer_count ? *K.defer_count * 32ull : (unsigned long long)m;
    const unsigned long long n_warps = (unsigned long long)gridDim.x * PC_KNN_WARPS;
    for (unsigned long long it = (unsigned long long)blockIdx.x * PC_KNN_WARPS + w; it < n_items; it += n_warps) {
        const long long t = K.defer_count ? (long long)K.defer_list[it >> 5] * 32 + (long long)(it & 31u) : (long long)it;
        if (t >= m_search) continue;
        uint32_t slot;
        float qx, qy, qz;
        pc_knn_fetch(q, qstride, perm, ordered, t, slot, qx, qy, qz);
        pc_knn_wlist W;
        W.ld = W.kd = INFINITY; W.li = W.ki = PC_KNN_NONE; W.thr = K.bound_thr;
        if (T.n_points > 0) pc_knn_warp_search(T, K, qx, qy, qz, s_front[w], lane, W);
        if (lane < K.k) {
            const size_t o = (size_t)slot * K.k + lane;
            if (out_idx) out_idx[o] = (int32_t)W.li;
            if (out_d2) out_d2[o] = (float)W.ld;
        }
        __syncwarp();
    }
}

// ---- warp packets of 32 curve-ordered queries ------------------------------------------------------------------------------
// Lane-private k-lists in dynamic shared memory, [entry][lane] so that the lanes of a warp never share a bank: per warp
// k x 32 doubles, then (after all warps' doubles) k x 32 indices -- 12 k bytes per query, 48 KB per CTA at k = 32.
__device__ __forceinline__ void pc_knn_lane_scan(const float4 *__restrict__ pts, uint32_t cnt, float qx, float qy, float qz,
                                                 const pc_knn_dev &K, double *__restrict__ Ld, uint32_t *__restrict__ Li,
                                                 double &kd, uint32_t &ki, float &thr)
{
#pragma unroll
    for (int i = 0; i < PC_LEAF; i++) {
        if ((uint32_t)i >= cnt) break;
        const float4 p = __ldg(pts + i);
        const float dx = p.x - qx, dy = p.y - qy, dz = p.z - qz;
        if (!(fmaf(dz, dz, fmaf(dy, dy, dx * dx)) <= thr)) continue;
        const double e = pc_exact_d2(p.x, p.y, p.z, (double)qx, (double)qy, (double)qz);
        const uint32_t id = (uint32_t)__float_as_int(p.w);
        if (!(e <= K.r2) || !pc_knn_less(e, id, kd, ki)) continue;
        int j = K.k - 1;
        for (; j > 0; j--) {                             // insertion into the sorted column
            const double dj = Ld[(j - 1) * 32];
            const uint32_t ij = Li[(j - 1) * 32];
            if (!pc_knn_less(e, id, dj, ij)) break;
            Ld[j * 32] = dj; Li[j * 32] = ij;
        }
        Ld[j * 32] = e; Li[j * 32] = id;
        kd = Ld[(K.k - 1) * 32]; ki = Li[(K.k - 1) * 32];
        thr = fminf(K.bound_thr, pc_thr_from(kd));
    }
}

__global__ void __launch_bounds__(32 * PC_KNN_WARPS)
pc_knn_packet_kernel(pc_tree T, pc_knn_dev K, const float *__restrict__ q, int64_t m, int qstride,
                     const uint32_t *__restrict__ perm, const float4 *__restrict__ ordered, const unsigned long long *__restrict__ m_eff,
                     int32_t *__restrict__ out_idx, float *__restrict__ out_d2)
{
    extern __shared__ double s_knn[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long m_search = m_eff ? (long long)*m_eff : (long long)m;
    const long long warp_id = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long t = warp_id * 32 + lane;
    if (warp_id * 32 >= m_search) return;                    // whole warp past the end
    double *Ld = s_knn + (size_t)w * K.k * 32 + lane;
    uint32_t *Li = reinterpret_cast<uint32_t *>(s_knn + (size_t)PC_KNN_WARPS * K.k * 32) + (size_t)w * K.k * 32 + lane;
    for (int j = 0; j < K.k; j++) { Ld[j * 32] = INFINITY; Li[j * 32] = PC_KNN_NONE; }
    const bool valid = t < m_search;
    uint32_t slot = 0;
    float qx = 0.f, qy = 0.f, qz = 0.f;
    if (valid) pc_knn_fetch(q, qstride, perm, ordered, t, slot, qx, qy, qz);
    double kd = INFINITY;
    uint32_t ki = PC_KNN_NONE;
    float thr = (valid && T.n_points > 0) ? K.bound_thr : -1.0f;     // thr < 0: this lane takes part in the votes only
    if (K.packet_split > 0.f) {
        // the incoherent-packet test of pc_query_packet_kernel: a packet with a query farther than packet_split (Chebyshev)
        // from its first one is answered by pc_knn_coop_kernel, one warp per query
        const float ax = __shfl_sync(PC_FULL_MASK, qx, 0), ay = __shfl_sync(PC_FULL_MASK, qy, 0), az = __shfl_sync(PC_FULL_MASK, qz, 0);
        const bool far = thr >= 0.f && fmaxf(fmaxf(fabsf(qx - ax), fabsf(qy - ay)), fabsf(qz - az)) > K.packet_split;
        if (__any_sync(PC_FULL_MASK, far)) {
            if (lane == 0) K.defer_list[atomicAdd(K.defer_count, 1ull)] = (uint32_t)warp_id;
            return;
        }
    }
    // the walk of pc_packet_traverse<1>: ballot on wanted children, majority vote for the nearer one, one stack per warp in
    // local memory at a warp-uniform index; leaves are scanned over their own counts
    if (__ballot_sync(PC_FULL_MASK, thr >= 0.f)) {
        if (T.root & PC_REF_LEAF) {
            pc_knn_lane_scan(T.points + (T.root & ~PC_REF_LEAF), T.root_count, qx, qy, qz, K, Ld, Li, kd, ki, thr);
        } else {
            uint32_t stack[PC_STACK];
            int sp = 0;
            uint32_t ref = T.root;
            for (;;) {
                const pc_rec rec = pc_load_rec(T.rec + 4ull * ref);
                const float2 dd = pc_rec_d2(rec, qx, qy, qz);
                const float d0 = dd.x, d1 = dd.y;
                const uint32_t w0 = __ballot_sync(PC_FULL_MASK, d0 <= thr), w1 = __ballot_sync(PC_FULL_MASK, d1 <= thr);
                uint32_t next = PC_NO_NODE;
                if (w0 | w1) {
                    const bool both = w0 != 0 && w1 != 0;
                    bool first0 = w1 == 0;
                    if (both) {
                        const uint32_t ia = __ballot_sync(PC_FULL_MASK, d0 <= thr || d1 <= thr);
                        const uint32_t pa = __ballot_sync(PC_FULL_MASK, d0 <= d1) & ia;
                        first0 = 2 * __popc(pa) >= __popc(ia);
                    }
                    const uint32_t r0 = pc_rec_ref(rec, 0), r1 = pc_rec_ref(rec, 1);
                    const uint32_t rn = first0 ? r0 : r1, rf = first0 ? r1 : r0;
                    const uint32_t cn = pc_rec_cnt(rec, first0 ? 0 : 1), cf = pc_rec_cnt(rec, first0 ? 1 : 0);
                    if (rn & PC_REF_LEAF) {
                        if ((first0 ? d0 : d1) <= thr) pc_knn_lane_scan(T.points + (rn & ~PC_REF_LEAF), cn, qx, qy, qz, K, Ld, Li, kd, ki, thr);
                    } else next = rn;
                    if (both) {
                        if (rf & PC_REF_LEAF) {
                            if ((first0 ? d1 : d0) <= thr) pc_knn_lane_scan(T.points + (rf & ~PC_REF_LEAF), cf, qx, qy, qz, K, Ld, Li, kd, ki, thr);
                        } else if (next != PC_NO_NODE) {
                            stack[sp] = rf;
                            sp++;
                        } else next = rf;
                    }
                }
                __syncwarp();
                if (next != PC_NO_NODE) { ref = next; continue; }
                if (sp == 0) break;
                sp--;
                ref = stack[sp];
            }
        }
    }
    if (valid) {
        const size_t o = (size_t)slot * K.k;
        for (int j = 0; j < K.k; j++) {
            if (out_idx) out_idx[o + j] = (int32_t)Li[j * 32];
            if (out_d2) out_d2[o + j] = (float)Ld[j * 32];
        }
    }
}
