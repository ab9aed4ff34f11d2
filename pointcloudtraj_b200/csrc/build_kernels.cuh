// build_kernels.cuh -- index construction kernels: bounding box, curve keys, prefix-split tree (nodes + bottom-up box fit).
//
// Index layout in HBM: ONE float4 array (`tree`) per index,
//   records tree[0 .. 4 (n-1))   : inner node i of the binary radix tree over the curve-sorted keys (T. Karras, HPG 2012) is the
//                                  64-byte record tree[4i .. 4i+3], the tight boxes of its two children with the two children
//                                  INTERLEAVED per axis, as 16 words:
//                                    [min0.x min1.x min0.y min1.y min0.z min1.z ref0 ref1 | max0.x max1.x max0.y max1.y max0.z max1.z cnt0 cnt1]
//                                  (ref = child reference, cnt = number of points when the child is a leaf), so that a
//                                  256-bit load puts (child 0, child 1) of one bound into adjacent registers and one packed
//                                  fp32x2 instruction handles both children (query_kernels.cuh).  Every node is split where
//                                  the highest differing bit of its first and last key flips, so node boundaries coincide
//                                  with the cells of the curve.
//   points  tree[4 (n-1) .. +n+PC_LEAF) : (x, y, z, original index as int bits) in curve order, padded with PC_LEAF copies of
//                                  the last point (a leaf scan reads PC_LEAF consecutive points from any start).
// A child whose range holds <= PC_LEAF points is a LEAF: its reference is PC_REF_LEAF | (index of its first point).  Inner
// nodes whose own range is that small are never referenced and their records stay unwritten.  A cloud of <= PC_LEAF points
// has no inner node: the root reference is the leaf PC_REF_LEAF | 0.
// A traversal step loads the record of the node it visits (two 256-bit loads) or the four points of a leaf.
// replaces struct kdtree / struct kdnode / struct kdhyperrect (Utils/kdtree/src/kdtree.c:56-80), insert_rec (:167-194) and
// hyperrect_extend (kdtree.c:729-741).
#pragma once
#include "common.cuh"
#define PC_LBVH_LEAF PC_LEAF
#include "lbvh.cuh"

#define PC_BUILD_THREADS 256

// ---- bounding box of the cloud: bbox[0..2] = ordered(min), bbox[3..5] = ordered(max) ----------------
// Only points whose three coordinates are all finite count: one infinite coordinate would make the extent infinite, the
// cell size zero and every key 0 (the tree would follow the input order).  Points with a NaN or an infinity are still
// indexed; their cells clamp to the frame.  A cloud without a finite point keeps the initial +inf / -inf.
__global__ void __launch_bounds__(PC_BUILD_THREADS)
pc_bbox_kernel(const float *__restrict__ xyz, int64_t n, int stride, uint32_t *__restrict__ bbox)
{
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float *p = xyz + i * stride;
        const float x = p[0], y = p[1], z = p[2];
        if (!(isfinite(x) && isfinite(y) && isfinite(z))) continue;
        lo[0] = fminf(lo[0], x); lo[1] = fminf(lo[1], y); lo[2] = fminf(lo[2], z);
        hi[0] = fmaxf(hi[0], x); hi[1] = fmaxf(hi[1], y); hi[2] = fmaxf(hi[2], z);
    }
#pragma unroll
    for (int a = 0; a < 3; a++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(PC_FULL_MASK, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(PC_FULL_MASK, hi[a], o));
        }
    }
    __shared__ float s_lo[PC_BUILD_THREADS / 32][3], s_hi[PC_BUILD_THREADS / 32][3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; a++) { s_lo[warp][a] = lo[a]; s_hi[warp][a] = hi[a]; }
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        int a = threadIdx.x;
        float l = s_lo[0][a], h = s_hi[0][a];
        for (int w = 1; w < PC_BUILD_THREADS / 32; w++) { l = fminf(l, s_lo[w][a]); h = fmaxf(h, s_hi[w][a]); }
        atomicMin(&bbox[a], pc_float_to_ordered(l));
        atomicMax(&bbox[3 + a], pc_float_to_ordered(h));
    }
}

// decode the bbox into the quantisation frame (device-side, no host round trip)
__device__ __forceinline__ pc_frame pc_make_frame(const uint32_t *bbox, int bits)
{
    pc_frame f;
    float ext = 0.0f;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        float lo = pc_ordered_to_float(bbox[a]), hi = pc_ordered_to_float(bbox[3 + a]);
        f.lo[a] = lo;
        ext = fmaxf(ext, hi - lo);
    }
    f.max_cell = (1u << bits) - 1u;
    // cells of edge ext / 2^bits; a degenerate cloud (ext == 0) maps everything to cell 0
    f.inv_cell = (ext > 0.0f && ext < INFINITY) ? ((float)(1u << bits) * (1.0f - 1e-6f)) / ext : 0.0f;
    return f;
}

// Order of the cloud along a space-filling curve.  Every prefix of a Hilbert key is a box of cells (an octant, two adjacent
// octants or a 2x2x1 slab of them), so the radix tree's nodes are compact; the same curve orders the query batches.
#ifndef PC_POINT_CURVE
#define PC_POINT_CURVE 1     // 0 = Morton, 1 = Hilbert
#endif
template <typename KeyT>
__global__ void __launch_bounds__(PC_BUILD_THREADS)
pc_keygen_kernel(const float *__restrict__ xyz, int64_t n, int stride, const uint32_t *__restrict__ bbox, int bits,
                 KeyT *__restrict__ keys, uint32_t *__restrict__ vals, uint32_t *__restrict__ ghist, int hist_passes)
{
    // ghist (nullable): digit histograms of all hist_passes sort passes (onesweep path of radix_sort.cuh), counted while the
    // key is in a register
    __shared__ uint32_t s_hist[8][256];
    if (ghist) {
        for (int j = threadIdx.x; j < hist_passes * 256; j += PC_BUILD_THREADS) (&s_hist[0][0])[j] = 0;
        __syncthreads();
    }
    const pc_frame f = pc_make_frame(bbox, bits);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float *p = xyz + i * stride;
#if PC_POINT_CURVE == 1
        if (sizeof(KeyT) == 4) keys[i] = (KeyT)pc_hilbert30(p[0], p[1], p[2], f);
        else keys[i] = (KeyT)pc_hilbert63(p[0], p[1], p[2], f, bits);
#else
        if (sizeof(KeyT) == 4) keys[i] = (KeyT)pc_morton30(p[0], p[1], p[2], f);
        else keys[i] = (KeyT)pc_morton63(p[0], p[1], p[2], f);
#endif
        vals[i] = (uint32_t)i;
        if (ghist) {
            const KeyT k = keys[i];
            for (int p = 0; p < hist_passes; p++) atomicAdd(&s_hist[p][(uint32_t)(k >> (8 * p)) & 255u], 1u);
        }
    }
    if (ghist) {
        __syncthreads();
        for (int j = threadIdx.x; j < hist_passes * 256; j += PC_BUILD_THREADS) {
            const uint32_t c = (&s_hist[0][0])[j];
            if (c) atomicAdd(&ghist[j], c);
        }
    }
}

// ---- tree, step 1: one thread per point slot ---------------------------------------------------------------------------------
// Thread i gathers point order[i] into curve position i and, for i < n - 1, computes inner node i of the radix tree from the
// sorted keys: range, split, child references (the .w words of its record) and the parent links of its inner children.
// The arrival counters of the fit kernel are cleared here.
#define PC_NODE_UNUSED 0xffffffffu
// word offsets inside a record (see the layout above); child slot c = 0 / 1
#define PC_REC_LO(axis, c) (2 * (axis) + (c))
#define PC_REC_HI(axis, c) (8 + 2 * (axis) + (c))
#define PC_REC_REF(c) (6 + (c))
#define PC_REC_CNT(c) (14 + (c))
#ifndef PC_FIT_ACQREL
#define PC_FIT_ACQREL 1             // arrival counter: one acq_rel atomic instead of fence + atomic + fence (-8 % build time)
#endif

template <typename KeyT>
__global__ void __launch_bounds__(PC_BUILD_THREADS)
pc_tree_nodes_kernel(const float *__restrict__ xyz, int stride, const uint32_t *__restrict__ order, const KeyT *__restrict__ keys,
                     int64_t n, float4 *__restrict__ rec, float4 *__restrict__ points, int32_t *__restrict__ parent,
                     int *__restrict__ arrived)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n + PC_LEAF) return;
    {
        const uint32_t src = order[i < n ? i : n - 1];                 // the pad slots repeat the last point
        const float *p = xyz + (int64_t)src * stride;
        points[i] = make_float4(p[0], p[1], p[2], __uint_as_float(src));
    }
    if (i >= n - 1 || n <= PC_LEAF) return;
    if (i == 0) parent[0] = -1;
    arrived[i] = 0;
    int64_t f, l, s;
    pc_lbvh_node(keys, n, i, &f, &l, &s);
    float *w = reinterpret_cast<float *>(rec + 4 * i);
    if (l - f + 1 <= PC_LEAF) { w[PC_REC_REF(0)] = __uint_as_float(PC_NODE_UNUSED); return; }   // collapsed into a leaf of its parent
    uint32_t r0, c0, r1, c1;
    pc_lbvh_children(f, l, s, &r0, &c0, &r1, &c1);
    w[PC_REC_REF(0)] = __uint_as_float(r0); w[PC_REC_CNT(0)] = __uint_as_float(c0);
    w[PC_REC_REF(1)] = __uint_as_float(r1); w[PC_REC_CNT(1)] = __uint_as_float(c1);
    if (!(r0 & PC_REF_LEAF)) parent[r0] = (int32_t)i;
    if (!(r1 & PC_REF_LEAF)) parent[r1] = (int32_t)i;
}

__device__ __forceinline__ void pc_leaf_box(const float4 *__restrict__ points, uint32_t first, uint32_t count, float *lo, float *hi)
{
    float lx = INFINITY, ly = INFINITY, lz = INFINITY, hx = -INFINITY, hy = -INFINITY, hz = -INFINITY;
    for (uint32_t k = 0; k < count; k++) {
        const float4 p = points[first + k];
        lx = fminf(lx, p.x); ly = fminf(ly, p.y); lz = fminf(lz, p.z);      // fminf / fmaxf ignore NaN coordinates
        hx = fmaxf(hx, p.x); hy = fmaxf(hy, p.y); hz = fmaxf(hz, p.z);
    }
    lo[0] = lx; lo[1] = ly; lo[2] = lz; hi[0] = hx; hi[1] = hy; hi[2] = hz;
}

// ---- tree, step 2: bottom-up box fit -------------------------------------------------------------------------------------------
// A CTA owns 256 consecutive node ids.  The subtree of a node covers a contiguous range of ids, so most of the lower levels
// live inside one CTA: phase A fits them in SHARED memory -- every node keeps the boxes of its two children there, a node is
// complete once both are known, and in rounds (one barrier each, about the depth of a 256-point subtree) a complete child's
// merged box moves into its parent's slot.  Phase B is the classic scheme for what is left (nodes whose children sit in other
// CTAs): a thread that completes a node writes its merged box into the parent's record and bumps the parent's arrival
// counter with one acquire-release atomic; whoever brings the counter to 2 carries on upwards from global memory.  Only the
// upper ~1 % of the nodes take the atomic path (the first version ran every level through it: 42 % of the build).
#define PC_FIT_THREADS 256

__global__ void __launch_bounds__(PC_FIT_THREADS)
pc_tree_fit_kernel(float4 *rec, const float4 *__restrict__ points, const int32_t *__restrict__ parent, int *arrived, int64_t n)
{
    __shared__ float s_box[PC_FIT_THREADS][2][6];          // [node][child slot][min xyz, max xyz]
    __shared__ unsigned char s_done[PC_FIT_THREADS];
    const int t = threadIdx.x;
    const int64_t B = (int64_t)blockIdx.x * PC_FIT_THREADS, i = B + t;
    const bool exists = i < n - 1;
    volatile float *w = reinterpret_cast<volatile float *>(rec + 4 * (exists ? i : 0));
    uint32_t r0 = PC_NODE_UNUSED, c0 = 0, r1 = 0, c1 = 0;
    if (exists) r0 = __float_as_uint(w[PC_REC_REF(0)]);
    const bool used = exists && r0 != PC_NODE_UNUSED;
    bool filled0 = false, filled1 = false;
    if (used) {
        c0 = __float_as_uint(w[PC_REC_CNT(0)]); r1 = __float_as_uint(w[PC_REC_REF(1)]); c1 = __float_as_uint(w[PC_REC_CNT(1)]);
        if (r0 & PC_REF_LEAF) { pc_leaf_box(points, r0 & ~PC_REF_LEAF, c0, &s_box[t][0][0], &s_box[t][0][3]); filled0 = true; }
        if (r1 & PC_REF_LEAF) { pc_leaf_box(points, r1 & ~PC_REF_LEAF, c1, &s_box[t][1][0], &s_box[t][1][3]); filled1 = true; }
    }
    s_done[t] = used && filled0 && filled1;
    // ---- phase A: rounds inside the CTA ----------------------------------------------------------------------------------
    const bool local0 = used && !(r0 & PC_REF_LEAF) && (int64_t)r0 >= B && (int64_t)r0 < B + PC_FIT_THREADS;
    const bool local1 = used && !(r1 & PC_REF_LEAF) && (int64_t)r1 >= B && (int64_t)r1 < B + PC_FIT_THREADS;
    for (;;) {
        __syncthreads();
        bool progress = false;
        if (used && !s_done[t]) {
#pragma unroll
            for (int c = 0; c < 2; c++) {
                const bool filled = c ? filled1 : filled0, local = c ? local1 : local0;
                if (!filled && local) {
                    const int ct = (int)((int64_t)(c ? r1 : r0) - B);
                    if (s_done[ct]) {
#pragma unroll
                        for (int k = 0; k < 3; k++) {
                            s_box[t][c][k] = fminf(s_box[ct][0][k], s_box[ct][1][k]);
                            s_box[t][c][3 + k] = fmaxf(s_box[ct][0][3 + k], s_box[ct][1][3 + k]);
                        }
                        if (c) filled1 = true; else filled0 = true;
                        progress = true;
                    }
                }
            }
        }
        // a node completed in this round becomes visible to its parent in the next one
        const bool now_done = used && filled0 && filled1;
        if (!__syncthreads_or(progress)) break;
        if (now_done) s_done[t] = 1;
    }
    if (!used) return;
    // the slots known so far go to the node's record (the others belong to children in other CTAs)
#pragma unroll
    for (int c = 0; c < 2; c++) {
        if (c ? filled1 : filled0) {
#pragma unroll
            for (int a = 0; a < 3; a++) { w[PC_REC_LO(a, c)] = s_box[t][c][a]; w[PC_REC_HI(a, c)] = s_box[t][c][3 + a]; }
        }
    }
    // ---- phase B: arrivals across CTAs ---------------------------------------------------------------------------------------
    // Every used node announces the slots it filled to its own counter; a node that is complete and whose parent did NOT take
    // its box in phase A (the parent sits in another CTA) pushes the box upwards.
    int add = (filled0 ? 1 : 0) + (filled1 ? 1 : 0);
    int64_t node = i;
    if (add == 2) {
        // complete inside the CTA: was the box consumed by a parent in this CTA?
        const int32_t par = parent[node];
        if (par < 0) return;                                                         // the root
        if ((int64_t)par >= B && (int64_t)par < B + PC_FIT_THREADS) return;        // yes (phase A ran until no progress was left)
    }
    while (add > 0) {
        if (!(node == i && add == 2)) {
            int old;
#if PC_FIT_ACQREL
            asm volatile("atom.acq_rel.gpu.global.add.s32 %0, [%1], %2;" : "=r"(old) : "l"(arrived + node), "r"(add) : "memory");
#else
            __threadfence();
            old = atomicAdd(&arrived[node], add);
            __threadfence();
#endif
            if (old + add < 2) break;                          // another child's thread completes this node
        }
        const int32_t par = parent[node];
        if (par < 0) break;                                    // the root is complete
        volatile float *c = reinterpret_cast<volatile float *>(rec + 4 * node);
        volatile float *p = reinterpret_cast<volatile float *>(rec + 4 * (int64_t)par);
        const int slot = __float_as_uint(p[PC_REC_REF(0)]) == (uint32_t)node ? 0 : 1;     // left child = first reference of the parent
#pragma unroll
        for (int a = 0; a < 3; a++) {
            p[PC_REC_LO(a, slot)] = fminf(c[PC_REC_LO(a, 0)], c[PC_REC_LO(a, 1)]);
            p[PC_REC_HI(a, slot)] = fmaxf(c[PC_REC_HI(a, 0)], c[PC_REC_HI(a, 1)]);
        }
        node = par;
        add = 1;
    }
}

// ---- tree, step 3: seeds for the lane-group walks ------------------------------------------------------------------------------
// The kernels that put a whole group of lanes on ONE query (pc_query_coop_kernel, pc_range_coop_kernel) would spend their first
// five steps with 1, 2, 4, 8, 16 busy lanes if they started at the root.  One warp expands the top of the tree breadth-first
// until the next level would not fit 32 lanes and leaves the frontier here: up to 32 inner nodes, plus the (rare) leaves met
// on the way as (reference, count) pairs.  Layout (uint32 words): [0] inner count, [1] leaf count, [2..34) inner nodes,
// [34..98) leaf pairs.  Lives right behind the points, inside the span pc_index_broadcast ships.
#define PC_SEED_WORDS 100
#define PC_SEED_INNER 2
#define PC_SEED_LEAF 34

__global__ void __launch_bounds__(32)
pc_tree_seed_kernel(const float4 *__restrict__ rec, uint32_t root, uint32_t root_count, uint32_t *__restrict__ seeds)
{
    __shared__ uint32_t cur[32], nxt[64], leaf[64];
    const int lane = threadIdx.x;
    int n = 0, n_leaf = 0;
    if (root & PC_REF_LEAF) { if (lane == 0) { leaf[0] = root; leaf[1] = root_count; } n_leaf = 1; }
    else { if (lane == 0) cur[0] = root; n = 1; }
    __syncwarp();
    while (n > 0 && 2 * n <= 32 && n_leaf + 2 * n <= 32) {
        uint32_t r[2] = { 0, 0 }, c[2] = { 0, 0 };
        bool inner[2] = { false, false }, isleaf[2] = { false, false };
        if (lane < n) {
            const float *w = reinterpret_cast<const float *>(rec + 4ull * cur[lane]);
            r[0] = __float_as_uint(w[PC_REC_REF(0)]); c[0] = __float_as_uint(w[PC_REC_CNT(0)]);
            r[1] = __float_as_uint(w[PC_REC_REF(1)]); c[1] = __float_as_uint(w[PC_REC_CNT(1)]);
            for (int k = 0; k < 2; k++) { isleaf[k] = (r[k] & PC_REF_LEAF) != 0; inner[k] = !isleaf[k]; }
        }
        int n_new = 0;
        const uint32_t lt = (1u << lane) - 1u;
        for (int k = 0; k < 2; k++) {
            const uint32_t mi = __ballot_sync(PC_FULL_MASK, inner[k]), ml = __ballot_sync(PC_FULL_MASK, isleaf[k]);
            if (inner[k]) nxt[n_new + __popc(mi & lt)] = r[k];
            if (isleaf[k]) { const int p = n_leaf + __popc(ml & lt); leaf[2 * p] = r[k]; leaf[2 * p + 1] = c[k]; }
            n_new += __popc(mi);
            n_leaf += __popc(ml);
        }
        __syncwarp();
        if (lane < n_new) cur[lane] = nxt[lane];
        n = n_new;
        __syncwarp();
    }
    if (lane == 0) { seeds[0] = (uint32_t)n; seeds[1] = (uint32_t)n_leaf; }
    if (lane < n) seeds[PC_SEED_INNER + lane] = cur[lane];
    if (lane < n_leaf) { seeds[PC_SEED_LEAF + 2 * lane] = leaf[2 * lane]; seeds[PC_SEED_LEAF + 2 * lane + 1] = leaf[2 * lane + 1]; }
}
