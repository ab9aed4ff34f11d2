/*
 * pc_index.h -- C ABI of libpcindex.so: exact nearest-obstacle queries against a raw point cloud
 * on one NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary for pointcloudTraj's hot path.  Each entry point names the
 * reference interface it replaces (paths relative to the reference checkout):
 *
 *   pc_index_create / destroy   kd_create / kd_free                 Utils/kdtree/include/kdtree/kdtree.h:39-46
 *                                                                   (Utils/kdtree/src/kdtree.c:112-134)
 *   pc_index_build              kd_clear + n x kd_insert3(x,y,z,(void*)i)   kdtree.h:49,58  (kdtree.c:143-159,244-251)
 *                               == safeRegionRrtStar::setInput      Planner/src/corridor_finder.cpp:93-99
 *   pc_nearest_batch            kd_nearest3 + kd_res_item + kd_res_free     kdtree.h:67,113,97 (kdtree.c:493-500,641-650,613)
 *   pc_knn_batch                pcl::search::KdTree nearestKSearch, radiusSearch with max_nn (no counterpart in Utils/kdtree)
 *   pc_knn_large_batch          pcl::search::KdTree nearestKSearch with 32 < k <= 1024
 *   pc_segment_nearest_batch    (no counterpart: the reference samples points along an edge) nearest point to a segment
 *   pc_sphere_sweep_batch       (no counterpart: the reference checks sampled positions) first contact of a sphere moved
 *                               along a segment
 *   pc_range_batch              kd_nearest_range3 + kd_res_size/next/item   kdtree.h:92,100-113 (kdtree.c:595-602)
 *   pc_range_sorted_batch       pcl::search::KdTree radiusSearch(q, r, k_indices, k_sqr_distances, max_nn), any max_nn
 *   pc_radius_batch             safeRegionRrtStar::radiusSearch     Planner/src/corridor_finder.cpp:113-133
 *                               (parameters of setParam :17-23, start point of setStartPt :43-50)
 *   pc_clearance_batch          checkSafeTrajectory + getPosFromBezier + checkTrajPtCol
 *                               Planner/src/sim_planning_demo.cpp:729-781, :715-727; corridor_finder.cpp:412-416
 *   pc_trajectory_sweep_batch   (no counterpart: the reference samples every dt) certified first contact of a sphere moved
 *                               along a piecewise Bezier trajectory
 *   pc_trajectory_nearest_batch (no counterpart: the reference samples every dt) certified clearance of a piecewise Bezier
 *                               trajectory: its distance to the nearest cloud point to within tol, with a witness
 *   pc_distance_field           (no counterpart) the truncated distance field (ESDF) of the cloud on a voxel lattice, with
 *                               the nearest point of every voxel centre
 *   pc_comm_* / pc_index_broadcast   (no counterpart: the reference is single-process) -- replicate the
 *                               built index to the other GPUs of the host with one ncclBroadcast.
 *
 * Conventions (kept from the reference's C API): opaque handle created and destroyed by the
 * caller; int return, 0 = success, negative = error (never aborts, never throws); an empty index
 * is legal (kd_nearest3 returns NULL -> idx -1, d2 +inf); the caller owns every in/out buffer;
 * the index copies the cloud.  One host thread per handle.
 *
 * Memory spaces: every batch call takes `space` = PC_HOST or PC_DEVICE and ALL of its array
 * arguments live in that space.  PC_DEVICE calls are asynchronous on the handle's stream (call
 * pc_index_sync or synchronise the stream you passed to pc_index_create); PC_HOST calls return
 * when the results are in the caller's host buffers (pinned buffers from pc_host_alloc make the
 * copies asynchronous and pipelined with the kernels).  Blocking PC_HOST calls of up to 4096
 * queries -- the planner's own one-radiusSearch-per-iteration pattern -- take a low-latency path:
 * queries and results travel through mapped pinned memory and a whole warp works on each
 * search (about 20 us per single-query call, any host memory).  PC_HOST_ASYNC calls (pinned host buffers) only enqueue the
 * batch -- copy in, kernels, copy out -- on one of three internal streams in turn and return; results are valid after
 * pc_index_sync.  Back-to-back PC_HOST_ASYNC batches overlap their PCIe copies with each other's kernels; the caller
 * must give every batch in flight its own buffers.
 *
 * Exactness contract (DESIGN.md "Tie rule"): out_idx is the point that minimises the reference's
 * fp64 expression d2 = ((px-qx)^2 + (py-qy)^2) + (pz-qz)^2 (float32 inputs widened to double,
 * no FMA contraction); among several exact minimisers the LOWEST original index is returned.
 * out_d2 / out_radius are the fp64 values rounded once to float32.
 */
#ifndef PC_INDEX_H_
#define PC_INDEX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PC_OK          0
#define PC_EINVAL     (-1)  /* bad argument                                              */
#define PC_ENOMEM     (-2)  /* host or device allocation failed (kd_insert returns -1)   */
#define PC_ECUDA      (-3)  /* CUDA runtime error, see pc_last_error                     */
#define PC_ECAP       (-4)  /* output capacity too small; counts/offsets are still valid */
#define PC_ENCCL      (-5)  /* NCCL not available or NCCL error                          */
#define PC_ENOTIMPL   (-6)

#define PC_HOST   0
#define PC_DEVICE 1
#define PC_HOST_ASYNC 2   /* pc_nearest_batch / pc_radius_batch only: host buffers (pinned), the call returns at once */
#define PC_DEVICE_ASYNC 3 /* pc_nearest_batch / pc_radius_batch only: device buffers, batches rotate over three internal
                             streams (ordered after the handle's stream at call time); results valid after pc_index_sync */

/* flags for pc_radius_batch / pc_clearance_batch */
#define PC_RADIUS_BOUNDED   0  /* default: search only within max_radius + search_margin (exact for the radius) */
#define PC_RADIUS_FULL_NN   1  /* unbounded search: out_idx is the true nearest point even where the radius clamps */
/* flags for pc_nearest_batch / pc_radius_batch / pc_knn_batch / pc_knn_large_batch / pc_segment_nearest_batch /
 * pc_sphere_sweep_batch: reorder the batch along a space-filling (Hilbert) curve first (same results) */
#define PC_QUERY_AUTO      0
#define PC_QUERY_UNSORTED  2
#define PC_QUERY_SORTED    4

typedef struct pc_index pc_index;

/* safeRegionRrtStar::setParam (corridor_finder.cpp:17-23) + start_pt (corridor_finder.cpp:43-50).
 * sample_range < 0 disables the out-of-sensing-range early-out of radiusSearch (:115-116). */
typedef struct pc_radius_params {
    double search_margin;
    double max_radius;
    double sample_range;
    double start[3];
} pc_radius_params;

/* One piecewise Bezier trajectory = segments [first_seg, first_seg + num_seg) of the segment arrays;
 * t_now = max(0, odom stamp - trajectory start) of checkSafeTrajectory (sim_planning_demo.cpp:735). */
typedef struct pc_traj {
    int32_t first_seg;
    int32_t num_seg;
    double  t_now;
} pc_traj;

/* device-side layout of a built index (for inspection and for replication across GPUs): a binary radix tree over the
 * cloud sorted along a Hilbert curve, leaves of <= 4 consecutive points (pointcloudtraj_b200/csrc/build_kernels.cuh) */
typedef struct pc_index_view {
    int64_t n_points;      /* points in the cloud                                                            */
    int64_t n_nodes;       /* inner-node records: n_points - 1, or 0 when the whole cloud is one leaf          */
    uint32_t root;         /* child reference of the whole cloud: inner node 0, or 0x80000000 | 0 (a leaf)      */
    uint32_t root_count;   /* points of the root when it is a leaf                                            */
    const void *points;    /* float4[n_points + 4]: x, y, z, original index (int bits), curve order; = records + 4 n_nodes */
    const void *records;   /* float4[4 * n_nodes]: node i -> 16 words, the boxes of its two children interleaved per axis:
                              [min0.x min1.x min0.y min1.y min0.z min1.z ref0 ref1 | max0.x max1.x max0.y max1.y max0.z max1.z cnt0 cnt1]
                              ref = child reference (bit 31: leaf, low bits: first point), cnt = leaf point count       */
    float bbox_lo[3], bbox_hi[3];  /* per-axis min / max over the points whose x, y and z are all finite: the frame of the
                              curve keys.  Points with a NaN or infinite coordinate are indexed but do not widen it.  A cloud
                              without a finite point gives bbox_lo = +inf and bbox_hi = -inf; an empty index gives zeros  */
} pc_index_view;

/* ---- lifetime ------------------------------------------------------------------------------- */
int  pc_index_create(pc_index **out, int device, int64_t max_points, void *cuda_stream /* nullable */);
void pc_index_destroy(pc_index *ix);
int  pc_index_sync(pc_index *ix);                       /* wait for the handle's stream */
const char *pc_last_error(const pc_index *ix);          /* ix may be NULL: last create() failure */
const char *pc_version(void);

/* ---- index ---------------------------------------------------------------------------------- */
/* stride_floats = 3 (packed xyz) or 4 (pcl::PointXYZ / PointCloud2 x,y,z,pad layout). n == 0 is legal. */
int  pc_index_build(pc_index *ix, const float *xyz, int64_t n, int64_t stride_floats, int space);
int64_t pc_index_size(const pc_index *ix);
int  pc_index_view_get(const pc_index *ix, pc_index_view *out);
/* device time of the last pc_index_build on this handle, ms (CUDA events; syncs the stream) */
int  pc_index_last_build_ms(pc_index *ix, float *ms);

/* ---- queries -------------------------------------------------------------------------------- */
/* out_idx: -1 when the index is empty; out_d2: +inf when empty.  Either output may be NULL. */
int  pc_nearest_batch(pc_index *ix, const float *q_xyz, int64_t m, int64_t q_stride, int space, int flags,
                      int32_t *out_idx, float *out_d2);

/* out_radius = min(sqrt(d2) - search_margin, max_radius), or max_radius - search_margin for the
 * early-outs (query farther than sample_range + max_radius from start; empty index).
 * out_idx (nullable): nearest point, -1 for early-outs and (PC_RADIUS_BOUNDED) where the radius clamps. */
int  pc_radius_batch(pc_index *ix, const float *q_xyz, int64_t m, int64_t q_stride, int space, int flags,
                     const pc_radius_params *params, float *out_radius, int32_t *out_idx);

/* All points with d2 <= range^2 (inclusive, kdtree.c:273).  range: one value (range_is_scalar) or m values.
 * out_offsets[m+1] is the CSR row pointer; out_idx[cap] the concatenated lists (each list ascending by
 * original index).  If the total exceeds cap: returns PC_ECAP, out_offsets is still complete, out_idx untouched
 * beyond what fits.  Pass out_idx == NULL, cap == 0 to get the offsets only (returns PC_OK). */
int  pc_range_batch(pc_index *ix, const float *q_xyz, int64_t m, int64_t q_stride, int space,
                    const double *range, int range_is_scalar,
                    int64_t *out_offsets, int32_t *out_idx, int64_t cap);

/* pcl::search::KdTree::radiusSearch(q, r, k_indices, k_sqr_distances, max_nn) for a batch, exactly.  Row i holds the hit set
 * of pc_range_batch for the same (q, range) -- d2 <= range^2 in fp64, inclusive -- ascending by (fp64 d2, original index):
 * points at equal distance come lowest index first, the tie rule of pc_knn_batch.
 *   max_nn == 0   every hit;  max_nn > 0   the first max_nn entries of that order;  max_nn < 0   PC_EINVAL.
 * out_offsets[m+1] is the CSR row pointer over the row lengths min(hits, max_nn); out_idx[cap] the concatenated rows;
 * out_d2[cap] (nullable) each entry's fp64 d2 rounded once to float32, the value pc_knn_batch writes.  Capacity as for
 * pc_range_batch: a total above cap returns PC_ECAP with out_offsets complete; out_idx == NULL, out_d2 == NULL, cap == 0
 * returns the offsets only (PC_OK).  space: PC_HOST or PC_DEVICE (the ASYNC spaces return PC_EINVAL).  A pc_batch_shard
 * handle answers every query, as pc_range_batch does.  With a scalar range and max_nn <= PC_KNN_MAX a row equals the
 * non-padding prefix of pc_knn_batch(k = max_nn, max_range = range). */
int  pc_range_sorted_batch(pc_index *ix, const float *q_xyz, int64_t m, int64_t q_stride, int space,
                           const double *range, int range_is_scalar, int64_t max_nn,
                           int64_t *out_offsets, int32_t *out_idx, float *out_d2, int64_t cap);

/* The k nearest points of every query (pcl::search::KdTree::nearestKSearch; with a bound, radiusSearch(q, r, ..., max_nn = k)).
 * Row i is out_idx[i*k .. i*k+k) and out_d2[i*k .. i*k+k); either output may be NULL.  Entries are the k smallest points
 * under the lexicographic order (fp64 d2, original index), d2 the reference's expression of the exactness contract above:
 * among points tied at the k-th distance the lowest indices win, and at k = 1 this is the tie rule of pc_nearest_batch.
 * out_d2 holds the fp64 value rounded once to float32.
 *   max_range < 0    unbounded.
 *   max_range >= 0   only points with d2 <= max_range^2 (the inclusion test of pc_range_batch, max_range^2 in fp64): a
 *                    bounded row is the first k entries of pc_range_batch's list for the same range, re-sorted by (d2, index).
 * Rows with fewer than k points (small cloud, empty index, the bound) are padded with idx -1 and d2 +inf.
 * k in [1, PC_KNN_MAX], else PC_EINVAL; for more neighbours use pc_knn_large_batch (k <= PC_KNN_LARGE_MAX, bounded or
 * not) or pc_range_sorted_batch (bounded, any length).  space: PC_HOST or PC_DEVICE (the ASYNC
 * spaces return PC_EINVAL).  flags: PC_QUERY_AUTO / PC_QUERY_UNSORTED / PC_QUERY_SORTED as for pc_nearest_batch.  A handle
 * in pc_batch_shard mode (n_ranks > 1) returns PC_EINVAL.  k = 1 unbounded runs pc_nearest_batch. */
#define PC_KNN_MAX 32
int  pc_knn_batch(pc_index *ix, const float *q_xyz, int64_t m, int64_t q_stride, int space, int flags,
                  int k, double max_range, int32_t *out_idx, float *out_d2);

/* pcl::search::KdTree nearestKSearch(q, k) for 1 <= k <= PC_KNN_LARGE_MAX: the arguments, rows, order, bound, padding,
 * spaces and flags of pc_knn_batch, with longer rows.  Row i is out_idx[i*k .. i*k+k) / out_d2[i*k .. i*k+k) (either output
 * may be NULL): the k smallest points under (fp64 d2, original index), ties at the k-th distance to the lowest index, d2
 * rounded once to float32; max_range >= 0 keeps only points with d2 <= max_range^2 (pc_range_batch's test), max_range < 0
 * is unbounded, a NaN max_range returns PC_EINVAL; short rows are padded with idx -1 and d2 +inf.
 * k outside [1, PC_KNN_LARGE_MAX], the ASYNC spaces, unknown flags and a pc_batch_shard handle return PC_EINVAL; longer
 * bounded lists come from pc_range_sorted_batch.  k <= PC_KNN_MAX runs pc_knn_batch.  The first PC_KNN_MAX columns of a row
 * are pc_knn_batch's row for k = PC_KNN_MAX, and a bounded row is the row of pc_range_sorted_batch with max_nn = k. */
#define PC_KNN_LARGE_MAX 1024
int  pc_knn_large_batch(pc_index *ix, const float *q_xyz, int64_t m, int64_t q_stride, int space, int flags,
                        int k, double max_range, int32_t *out_idx, float *out_d2);

/* Nearest cloud point to each line segment [a_i, b_i] (float32 endpoints, stride 3 or 4, a and b in the same space).
 * Distance: A = a, B = b, P = p widened to double; D = B - A, W = P - A per axis; L2 = (Dx*Dx + Dy*Dy) + Dz*Dz,
 * s = (Wx*Dx + Wy*Dy) + Wz*Dz, every operation rounded to nearest, never fused:
 *   s <= 0 or L2 == 0   d2 = the reference's expression of P against A (the exactness contract above)
 *   s >= L2             d2 = the same against B
 *   otherwise           t = s / L2 (IEEE division), E = W - t*D per axis, d2 = (Ex*Ex + Ey*Ey) + Ez*Ez.
 * out_idx[i] is the point with the smallest d2, the lowest original index among exact ties; out_d2[i] that fp64 value
 * rounded once to float32.  A segment with a == b gives exactly pc_nearest_batch's (idx, d2) for the point a.
 *   max_range < 0    unbounded.
 *   max_range >= 0   only points with d2 <= max_range^2 (pc_range_batch's test); a row without one gets idx -1, d2 +inf.
 * An empty index gives idx -1, d2 +inf.  A segment with a non-finite endpoint coordinate gives idx -1 and d2 NaN (empty
 * index or not): a collision check `d2 < r*r` must treat NaN as "not checked", e.g. test !(d2 >= r*r).
 * A polyline of n points is checked with b_xyz = a_xyz + stride and m = n - 1 (the two arrays may overlap).
 * Either output may be NULL.  space: PC_HOST or PC_DEVICE.  flags: PC_QUERY_AUTO / PC_QUERY_UNSORTED / PC_QUERY_SORTED
 * (SORTED orders the segments along the curve by their midpoints first; same results).  PC_EINVAL: a bad stride, a NULL
 * a_xyz / b_xyz with m > 0, the ASYNC spaces, unknown flags, a NaN max_range, a pc_batch_shard handle (n_ranks > 1). */
int  pc_segment_nearest_batch(pc_index *ix, const float *a_xyz, const float *b_xyz, int64_t m, int64_t stride,
                              int space, int flags, double max_range, int32_t *out_idx, float *out_d2);

/* First contact of a sphere of radius `radius` moved from a_i to b_i: the smallest parameter t in [0, 1] at which a cloud
 * point lies in the sphere, and that point.  Per point p, with A, B, P widened to double, D, W, L2 and s exactly as in
 * pc_segment_nearest_batch, R2 = radius * radius (pc_range_batch's r2), every operation rounded to nearest, never fused,
 * sqrt and division IEEE:
 *   c0 = the reference's expression of P against A  (= (Wx*Wx + Wy*Wy) + Wz*Wz)
 *   c0 <= R2                                     t(p) = 0
 *   else if L2 != 0 and s > 0:  h = c0 - R2, disc = s*s - L2*h;
 *        disc >= 0 and t' = h / (s + sqrt(disc)) <= 1      t(p) = t'
 *   otherwise, if the reference's expression of P against B <= R2     t(p) = 1
 *   otherwise                                    p makes no contact.
 * out_idx[i] is the contacting point with the smallest (t(p), original index); out_t[i] that t rounded once toward -inf to
 * float32, so that a + out_t * (b - a) never passes the fp64 contact.  t = 0 exactly when pc_range_batch(a, radius) is
 * non-empty, and out_idx is then that list's first (lowest) index.  No contact, or an empty index: idx -1, t +inf.  A
 * non-finite endpoint coordinate: idx -1, t NaN.  A polyline of n points is checked with b_xyz = a_xyz + stride and
 * m = n - 1.  Either output may be NULL.  space: PC_HOST or PC_DEVICE.  flags as pc_segment_nearest_batch (SORTED orders by
 * the midpoints; same results).  PC_EINVAL: a radius that is negative, NaN or infinite, and every refusal of
 * pc_segment_nearest_batch (bad stride, NULL a_xyz / b_xyz with m > 0, the ASYNC spaces, unknown flags, pc_batch_shard). */
int  pc_sphere_sweep_batch(pc_index *ix, const float *a_xyz, const float *b_xyz, int64_t m, int64_t stride,
                           int space, int flags, double radius, int32_t *out_idx, float *out_t);

/* Arithmetic of the radiusSearch epilogue (pc_radius_batch, pc_clearance_batch) on this handle:
 *   PC_ARITH_FP64 (default)  radius = sqrt(d2) - search_margin in double precision from the kd-tree's fp64 d2 -- the parity
 *                            target the north star names (Utils/kdtree), within 1e-6 relative of the variant below;
 *   PC_ARITH_PCL_FLOAT       d2 rounded to float32, float32 sqrt, then the double subtraction: what corridor_finder.cpp:130-131
 *                            computes through PCL's interface (std::vector<float> k_sqr_distances; sqrt(float)).  Bit-identical
 *                            with the unmodified corridor_finder.cpp compiled against an exact 1-NN (tests/test_planner_ref*.py). */
#define PC_ARITH_FP64      0
#define PC_ARITH_PCL_FLOAT 1
int  pc_index_set_radius_arith(pc_index *ix, int mode);

/* Sensing gather: ALL points within `radius` of one centre (d2 <= radius^2; the centre is cast to float32 as PCL does),
 * ascending original index -- the LiDAR-mode observation of the reference's sensor node, one radiusSearch(pos, max_dist)
 * on the global map (Planner/src/camera_sensor.cpp:133-145).  *out_count (host) is always the number of hits; if it
 * exceeds cap the call returns PC_ECAP (cap == 0 with out_idx == NULL just counts). */
int  pc_sphere_gather(pc_index *ix, const double center[3], double radius, int space,
                      int32_t *out_idx, int64_t cap, int64_t *out_count);

/* Per trajectory: walk the segments from t_now in steps of dt while the accumulated time <= horizon
 * (sim_planning_demo.cpp:745-749), evaluate p = T_i * sum_j C(n,j) c_ij u^j (1-u)^(n-j), u = t/T_i,
 * cast to float32 and apply radiusSearch.  seg_coef_off[s] is the offset (in doubles) of segment s's
 * [x_0..x_n | y_0..y_n | z_0..z_n] block in coef; seg_order[s] = n in [1, 12].
 * out_first_hit[t]  : ordinal of the first sample with radius < 0 (the reference returns true there), -1 if none
 * out_min_radius[t] : min radiusSearch value over all samples within the horizon (+inf if no samples)
 * out_n_samples[t]  : samples within the horizon (nullable) */
int  pc_clearance_batch(pc_index *ix, const pc_traj *traj, int64_t n_traj,
                        const int32_t *seg_order, const double *seg_T, const int64_t *seg_coef_off,
                        int64_t n_seg, const double *coef, int64_t n_coef, int space,
                        double dt, double horizon, const pc_radius_params *params,
                        int32_t *out_first_hit, float *out_min_radius, int32_t *out_n_samples);

/* Certified first contact of a sphere of radius `radius` moved along each trajectory, in continuous time (not the dt walk of
 * pc_clearance_batch).  Trajectory arrays, their validation and their spaces as pc_clearance_batch.  Segment s (order
 * n = seg_order[s], duration T = seg_T[s]) is at local time sigma in [0, T] at the exact real value
 * C_s(sigma) = T * sum_j C(n,j) c_j u^j (1-u)^(n-j), u = sigma / T: the Bezier curve of the control points T * c_j.
 * The motion starts where pc_clearance_batch starts (t_s = max(0, t_now), then its fp64 segment-skipping loop: segment i0,
 * local time sigma0), covers the rest of segment i0 and the following segments of the trajectory in order, and stops where
 * the elapsed time reaches `horizon` (horizon == 0: the start point only; the end is rounded up, never cut short).  It is
 * empty when horizon < 0, when the trajectory has no segment, or when sigma0 > T on its last segment.
 * A cloud point p (float32 widened; non-finite points never touch) touches at (s, sigma) when |C_s(sigma) - p| <= radius.
 * With F(rho) the first such (segment, sigma) of the motion in time order at radius rho, the answer (out_seg[t], out_s[t],
 * out_idx[t]) = (s_c, sigma_c, i) satisfies
 *   1. nothing earlier: (s_c, sigma_c) <= F(radius) -- every point of the motion before it is farther than radius from the cloud;
 *   2. witness: |C_{s_c}(sigma_c) - p_i| <= radius + tol, so F(radius + tol) <= (s_c, sigma_c);
 *   3. complete: a contact is reported whenever F(radius) exists (with closest approach in (radius, radius + tol] either
 *      answer may come).
 * out_seg is an index into the segment arrays; out_s is rounded down so that rule 1 holds.  No contact (or an empty motion,
 * or an empty index): -1, +inf, -1.  A segment of the motion with a non-finite T or coefficient, or a control point T * c_j
 * beyond 1e37 in magnitude: -1, NaN, -1 ("not checked").  Deterministic: PC_HOST and PC_DEVICE, and repeated calls, give the
 * same bits.  Rule 2 is guaranteed for tol >= 2^-37 ((n + 1) S + radius) on the contact's segment, S = max_j |T * c_j|
 * (DESIGN.md §4.13); the subdivision depth is capped at 50 levels so that every call terminates, and a piece still undecided
 * there is reported at its start -- rule 1 holds, rule 2 may not (only below that tol).  Outputs are nullable.
 * PC_EINVAL: radius negative, NaN or infinite; tol not finite or <= 0; horizon NaN; every argument pc_clearance_batch refuses
 * (including its host-side validation of segment ranges, orders, offsets and T); the ASYNC spaces; a pc_batch_shard handle. */
int  pc_trajectory_sweep_batch(pc_index *ix, const pc_traj *traj, int64_t n_traj,
                               const int32_t *seg_order, const double *seg_T, const int64_t *seg_coef_off,
                               int64_t n_seg, const double *coef, int64_t n_coef, int space,
                               double horizon, double radius, double tol,
                               int32_t *out_seg, double *out_s, int32_t *out_idx);

/* Certified clearance of each trajectory: the distance from its motion to the nearest cloud point, to within tol, with a
 * witness.  Trajectory arrays, their validation, their spaces and the motion are those of pc_trajectory_sweep_batch.  Let D*
 * be the infimum of |C_s(sigma) - p| over the positions of the motion and the cloud points p with finite coordinates.  The
 * answer (out_seg[t], out_s[t], out_idx[t], out_dist[t]) = (s_c, sigma_c, i, d) satisfies
 *   1. witness: sigma_c lies in the motion's part of segment s_c and |C_{s_c}(sigma_c) - p_i| <= d, so D* <= d;
 *   2. certificate: D* >= d - tol -- nothing on the motion comes closer than d - tol to any cloud point;
 *   3. bound: max_range < 0 is unbounded (a witness whenever the index has a finite point within 2^60 m of the motion and the
 *      motion is not empty; farther points are never searched, bounded or not).  With
 *      max_range >= 0 a row without a witness means D* >= max_range, a reported row has d <= max_range + tol, and with
 *      max_range <= D* <= max_range + tol either answer may come.
 * No witness (under the bound, an empty motion, an empty index, no finite cloud point): -1, +inf, -1, +inf.  A segment of the
 * motion with a non-finite or unusable T, order or coefficient, or a control point T * c_j beyond 1e37 in magnitude: -1, NaN,
 * -1, NaN ("not checked").  Deterministic: PC_HOST and PC_DEVICE, and repeated calls, give the same bits.  Rule 2 is
 * guaranteed for tol >= 2^-37 ((n + 1) S + d) on every segment of the motion, S = max_j |T * c_j| (DESIGN.md §4.14); the
 * subdivision depth is capped at 50 levels so that every call terminates -- below that tol rule 1 holds, rules 2 and 3 may
 * not.  Outputs are nullable.  PC_EINVAL: max_range NaN; tol not finite or <= 0; horizon NaN; every argument
 * pc_clearance_batch refuses (including its host-side validation); the ASYNC spaces; a pc_batch_shard handle. */
int  pc_trajectory_nearest_batch(pc_index *ix, const pc_traj *traj, int64_t n_traj,
                                 const int32_t *seg_order, const double *seg_T, const int64_t *seg_coef_off,
                                 int64_t n_seg, const double *coef, int64_t n_coef, int space,
                                 double horizon, double max_range, double tol,
                                 int32_t *out_seg, double *out_s, int32_t *out_idx, double *out_dist);

/* A regular voxel lattice: nx x ny x nz cubic voxels of edge `voxel`, voxel (0, 0, 0) with its outer corner at origin. */
typedef struct pc_lattice {
    double  origin[3];   /* world position of the outer corner of voxel (0, 0, 0), finite */
    double  voxel;       /* edge length, finite and > 0 */
    int64_t dims[3];     /* nx, ny, nz >= 0 */
} pc_lattice;

/* The truncated (unsigned) Euclidean distance field of the cloud on a lattice: for every voxel, the nearest cloud point to its
 * centre and the distance to it.
 *   centre   voxel (i, j, k) = (i_0, i_1, i_2) has c_a = (float)(origin_a + ((double)i_a + 0.5) * voxel) on axis a, every fp64
 *            operation rounded to nearest and never fused, then rounded once to float32.
 *   layout   element v = i + nx * (j + ny * k) of out_dist[nx*ny*nz] and out_idx[nx*ny*nz]: x fastest, z slowest.
 *   index    out_idx[v] is the row pc_knn_batch(k = 1, max_range) returns for the centre: the lowest original index among the
 *            exact fp64 minimisers of d2 (the exactness contract above), -1 when no point counts.
 *   distance out_dist[v] = sqrt(d2) of that point, correctly rounded in fp64, then rounded once to float32; +inf where idx is -1.
 *   bound    max_range < 0 is unbounded; max_range >= 0 keeps only points with d2 <= max_range^2 in fp64 (pc_range_batch's
 *            test); +inf is accepted.
 * An empty index gives -1 / +inf everywhere.  An empty lattice (a dim 0) returns PC_OK and writes nothing.  Either output may
 * be NULL.  Repeated calls, and PC_HOST and PC_DEVICE, give the same bits.  PC_DEVICE is one kernel launch on the handle's
 * stream with no scratch memory; PC_HOST copies the field home in chunks of whole brick layers (PC_HOST_CHUNK_QUERIES voxels
 * each, about).  For a position x in the voxel of centre c the nearest point is at least out_dist - |x - c| away (c is the
 * float32 centre above, not the exact middle of the voxel).
 * PC_EINVAL: a NULL lat; a non-finite origin; a voxel that is not finite or <= 0; a negative dim; more than 2^40 voxels; a
 * non-empty lattice whose first or last centre on an axis is not finite in float32; a NaN max_range; the ASYNC spaces; a
 * pc_batch_shard handle (n_ranks > 1). */
int  pc_distance_field(pc_index *ix, const pc_lattice *lat, double max_range, int space, float *out_dist, int32_t *out_idx);

/* ---- the RRT* sample stream and one speculative expansion batch, generated on the device ----------- */
/* genSample's state (corridor_finder.cpp:333-358, the branches taken while no path is known: inform_status == false).
 * engine_state is the state of std::default_random_engine (= minstd_rand0; the reference seeds it with 0, :12, which the
 * standard maps to state 1): the next draw is 16807 * engine_state mod (2^31 - 1).  lo/hi are the bounds of rand_x, rand_y,
 * rand_z, in_lo/in_hi those of rand_x_in, rand_y_in, rand_z_in (setPt, :52-91). */
typedef struct pc_sampler {
    uint32_t engine_state, reserved;
    double goal_ratio, inlier_ratio;
    double end_pt[3];
    double lo[3], hi[3];
    double in_lo[3], in_hi[3];
} pc_sampler;
/* The next k samples of that stream, bit-identical with k calls of genSample() on libstdc++ (two draws per uniform double,
 * one or four uniforms per sample; the variable stride is resolved on the device, see sampler_kernels.cuh).  out_xyz: k x 3
 * doubles in `space` (PC_HOST or PC_DEVICE); *out_engine_state (host, nullable): the state to continue from (seed a host
 * engine with it).  The informed-ellipsoid branch (:361-378, libm calls) is not offered: generate those samples on the host. */
int  pc_sample_batch(pc_index *ix, const pc_sampler *sampler, int64_t k, int space, double *out_xyz, uint32_t *out_engine_state);

/* The frozen node set a speculative batch is steered against: centres (n x 3 doubles, Node::coord), radii (Node::radius) and
 * valid flags, in node-list order; host memory. */
typedef struct pc_node_set {
    int64_t n;
    const double *coord;
    const float *radius;
    const uint8_t *valid;
} pc_node_set;
typedef struct pc_candidate {      /* one new node the expansion loop would go on with */
    double center[3];              /* genNewNode's centre (corridor_finder.cpp:385-402) */
    float radius;                  /* radiusSearch(centre) */
    int32_t nearest;               /* the vertex it was steered from (index into the node set) */
} pc_candidate;
/* One batch of the expansion loop (SafeRegionExpansion, corridor_finder.cpp:720-731) without per-sample host traffic: the
 * next k samples of `sampler` are generated on the device, each is steered from its nearest vertex of `set` (findNearstVertex
 * on the float32 centres, exact fp64 distances; `nodes` is a second handle that holds the index of the node set and is
 * rebuilt here), radiusSearch answers the centres against `cloud`'s index, and only the candidates the loop would keep
 * (nearest vertex valid, centre z >= z_l, radius >= safety_margin, :726-731) come back, in sample order.  out: host memory,
 * cap entries; *out_count is always the number of candidates (PC_ECAP if it exceeds cap).  Both handles must live on the
 * same device; a pc_batch_shard handle on either side (n_ranks > 1) returns PC_EINVAL.  Identical, candidate for candidate, with k x genSample + pc_nearest_batch + steering on the host +
 * pc_radius_batch (tests/test_sampler_gpu.py). */
int  pc_expand_batch(pc_index *cloud, pc_index *nodes, const pc_node_set *set, const pc_sampler *sampler,
                     const pc_radius_params *params, double z_l, double safety_margin, int64_t k,
                     pc_candidate *out, int64_t cap, int64_t *out_count, uint32_t *out_engine_state);

/* ---- pinned host memory for PC_HOST calls ------------------------------------------------------ */
void *pc_host_alloc(int64_t bytes);
void  pc_host_free(void *p);

/* ---- multi-GPU (one process per GPU) ------------------------------------------------------------ */
#define PC_NCCL_UNIQUE_ID_BYTES 128
typedef struct pc_comm pc_comm;
int  pc_comm_unique_id(char id[PC_NCCL_UNIQUE_ID_BYTES]);           /* rank 0; ship the bytes to the other ranks */
int  pc_comm_init(pc_comm **out, int rank, int n_ranks, const char id[PC_NCCL_UNIQUE_ID_BYTES], int device);
void pc_comm_destroy(pc_comm *c);
/* Replicate root's built index (points + nodes + header) into every rank's handle: ncclBroadcast on the
 * handle's stream.  After it returns every rank answers queries against the same index. */
int  pc_index_broadcast(pc_index *ix, pc_comm *c, int root);
/* Spatial sharding of query batches: after pc_batch_shard(ix, rank, n_ranks) every pc_nearest_batch / pc_radius_batch on
 * this handle expects the SAME full batch on every rank and answers only this rank's share: the cubic cells of the index's
 * curve frame (at a level chosen on the device from the index's bounding box, the batch size and n_ranks, so that a cell holds
 * about a thousand queries, a rank gets a few hundred cells and all ranks agree) are dealt to the ranks by a hash of the
 * cell coordinates.  Every query is answered by
 * exactly one rank; entries of other ranks' queries are left untouched in the output arrays (pre-fill them, e.g. out_idx
 * with INT32_MIN, to tell them apart).  A rank's share is as dense in space as the whole batch and spread over the whole
 * map, which keeps the search efficient and balanced when one batch is split over many GPUs.  n_ranks = 1 switches back.
 * Needs the ordering pass (PC_EINVAL when PC_SORT_BITS=0 disabled it).
 * A PC_DEVICE call of >= 2^20 queries in this mode synchronises the handle's stream once, in the middle of the call (it
 * reads the size of the share back, 8 bytes, and sizes the sort and search launches by it; PC_SHARD_EXACT=0 keeps the call
 * fully asynchronous with launches sized for the whole batch); the pipelined spaces never do. */
int  pc_batch_shard(pc_index *ix, int rank, int n_ranks);
/* contiguous slice [begin, end) of m units owned by `rank` (queries or trajectories) */
void pc_shard_range(int64_t m, int rank, int n_ranks, int64_t *begin, int64_t *end);

/* ---- instrumentation -------------------------------------------------------------------------- */
/* number of kernels this library launched on the handle since the last reset (for bench.py's gpu_launches) */
int64_t pc_launch_count(const pc_index *ix, int reset);
/* When enabled, PC_DEVICE query batches record CUDA events around their two phases on the handle's stream;
 * pc_profile_last_batch waits for them and returns the device time of the curve ordering of the batch
 * (0 when the batch was not reordered) and of the search kernel, in ms. */
int  pc_profile_enable(pc_index *ix, int on);
int  pc_profile_last_batch(pc_index *ix, float *order_ms, float *search_ms);
/* Detail of that ordering pass (ms): out[0] clearing the sort scratch, out[1] the key kernel (curve keys, sensing-range
 * early-outs, compaction, digit histograms), out[2] the radix-sort passes. */
int  pc_profile_last_order_detail(pc_index *ix, float out[3]);
/* Number of warp packets of the last PC_DEVICE pc_nearest_batch (or PC_RADIUS_FULL_NN pc_radius_batch) on this handle that
 * were not walked as a packet because
 * their queries lay too far apart (a packet cut across a jump of the curve order, or across two cells of a pc_batch_shard
 * share): their queries were answered by one independent walk each (pc_query_deferred_kernel).  Waits for the batch. */
int  pc_profile_last_deferred_packets(pc_index *ix, int64_t *packets);

#ifdef __cplusplus
}
#endif
#endif /* PC_INDEX_H_ */
