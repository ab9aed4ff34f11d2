// pc_index.cu -- C ABI of libpcindex.so (see include/pc_index.h) and the host-side orchestration:
// arena management, stream ordering, the chunked H2D / kernel / D2H pipeline for PC_HOST calls.
//
// No CPU fallback exists: every entry point either launches the sm_100a kernels or returns an error.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <stdarg.h>
#include <math.h>
#include <dlfcn.h>
#include <new>

#include "../../include/pc_index.h"
#include "common.cuh"
#include "radix_sort.cuh"
#include "build_kernels.cuh"
#include "query_kernels.cuh"
#include "range_kernels.cuh"
#include "knn_kernels.cuh"
#include "knn_large_kernels.cuh"
#include "range_sorted_kernels.cuh"
#include "segment_kernels.cuh"
#include "sweep_kernels.cuh"
#include "clearance_kernels.cuh"
#include "traj_sweep_kernels.cuh"
#include "traj_nearest_kernels.cuh"
#include "field_kernels.cuh"
#include "sampler_kernels.cuh"

#define PC_VERSION_STRING "pcindex 0.2 (sm_100a)"
#define PC_PIPE_LANES 3                 // concurrent H2D / kernel / D2H chunks for PC_HOST calls
#define PC_HOST_CHUNK (1 << 20)         // queries per pipelined chunk (scripts/e2e_sweep.py, profiles/r2_e2e_chunk_sweep.txt: 1 Mi
                                        // without a ramp of smaller first chunks is the optimum for 10 M batches on the
                                        // round-2 kernels; round 1: 3 Mi with a ramp)
#define PC_TINY_BATCH 4096              // PC_HOST calls up to this size: one kernel reading / writing mapped pinned host buffers
#define PC_SORT_MIN_RADIUS 640000       // PC_QUERY_AUTO orders radius / nearest batches at least this large: below, one thread per
#define PC_SORT_MIN_NEAREST 360000      // query on the UNORDERED batch is faster on the prefix-split tree (profiles/r2_mid_batch_ab.txt)
#define PC_COOP_MAX_BATCH 24576         // unordered batches up to this size: a group of lanes per query (profiles/r2_small_batch_ab.txt)
#define PC_COOP_MAX_BATCH_UNBOUNDED 8192
#define PC_SHARD_EXACT_MIN (1 << 20)    // pc_batch_shard: batches at least this large read their share's size back (see pc_share_size)
#define PC_STAGE_BYTES ((int64_t)1 << 18)   // each half of ix->h_stage: a small PC_HOST call's inputs go in, its results come back

static thread_local char g_create_error[256] = "";

// per-lane scratch for query batches (device staging for PC_HOST calls, sort buffers for Morton-ordered batches)
struct pc_lane {
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    float *d_q = nullptr; int64_t q_cap = 0;                 // floats
    int32_t *d_i32 = nullptr; int64_t i32_cap = 0;
    float *d_f32 = nullptr; int64_t f32_cap = 0;
    uint32_t *keys_a = nullptr, *keys_b = nullptr, *vals_a = nullptr, *vals_b = nullptr; int64_t sort_cap = 0;
    uint32_t *tile_hist = nullptr; int64_t hist_cap = 0;
    uint32_t *digit_total = nullptr;
    unsigned long long *counter = nullptr;                   // [1]: queries that still need a search after the ordering pass
    uint32_t *bins = nullptr; int64_t bins_cap = 0;          // cell-binning ordering: 2^bits counters / cursors + their tile sums
    float4 *ordered = nullptr; int64_t ordered_cap = 0;      // cell-binning ordering: the batch gathered into cell order
    float4 *d_mid = nullptr; int64_t mid_cap = 0;            // pc_segment_nearest_batch: the segments' midpoints (ordering keys)
    double per_cell = 0.0;                                   // last ordered batch: estimated queries per 1/256-extent cell
    cudaEvent_t done = nullptr;
    cudaStream_t order_stream = nullptr;                     // high-priority stream for the ordering pass of pipelined batches
    cudaStream_t os = nullptr;                               // stream the current batch's ordering pass runs on
    cudaEvent_t ev_deps = nullptr, ev_ordered = nullptr;
    cudaEvent_t t0 = nullptr, t1 = nullptr, t2 = nullptr;   // profiling: batch start / ordered / searched
    cudaEvent_t ta = nullptr, tb = nullptr;                 // profiling detail: scratch cleared / keys made (then the sort up to t1)
};

struct pc_index {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;

    // cloud / index
    int64_t cap = 0;          // points the arena can hold
    int64_t n = 0, n_nodes = 0;   // points, inner-node records (n - 1, or 0 when the cloud is a single leaf)
    uint32_t root = PC_REF_LEAF, root_count = 0;
    int key_bytes = 4;
    float *d_xyz = nullptr;   // staging copy of the caller's cloud for PC_HOST builds (cap * 4 floats)
    uint32_t *d_bbox = nullptr;
    void *keys_a = nullptr, *keys_b = nullptr;
    uint32_t *vals_a = nullptr, *vals_b = nullptr;
    uint32_t *tile_hist = nullptr; int64_t hist_cap = 0;
    uint32_t *digit_total = nullptr;
    float4 *tree = nullptr; int64_t tree_cap = 0;   // one allocation: records [0, 4 n_nodes) then points [4 n_nodes, + n + PC_LEAF)
    float4 *points = nullptr;                       // = tree + 4 n_nodes of the current build
    cudaEvent_t ev_b0 = nullptr, ev_b1 = nullptr, ev_ready = nullptr, ev_in = nullptr;
    uint32_t *h_bbox = nullptr;                      // pinned host copy of d_bbox, valid once ev_b1 has completed
    bool build_timed = false;
    bool bbox_from_bcast = false;                    // h_bbox was filled by pc_index_broadcast (receiver side)

    pc_lane lane[PC_PIPE_LANES];

    // generic device scratch for range / clearance / expansion batches
    void *scratch = nullptr; int64_t scratch_cap = 0;
    // pc_range_sorted_batch: the lists too long for the capturing warp, untruncated (fp64 d2, then original index)
    uint32_t *range_long = nullptr; int64_t range_long_cap = 0;
    // pinned staging block of small PC_HOST calls (pc_stage_upload): 2 * PC_STAGE_BYTES, inputs in the first half, results in the second
    char *h_stage = nullptr;
    // pc_expand_batch: running candidate totals per chunk (pinned) and the events the host waits on before copying a chunk back
    unsigned long long *h_totals = nullptr;
    cudaEvent_t ev_chunk[2] = { nullptr, nullptr };

    // tiny PC_HOST batches (the planner's one-query-at-a-time calls): pinned, device-mapped host buffers the kernel reads the
    // queries from and writes the results to directly -- one launch + one stream sync instead of two staged copies
    float *tiny_q = nullptr, *tiny_f = nullptr; int32_t *tiny_i = nullptr;          // host addresses
    float *tiny_q_dev = nullptr, *tiny_f_dev = nullptr; int32_t *tiny_i_dev = nullptr;   // the same memory as the device sees it

    int64_t launches = 0;
    bool profile = false, profiled = false;
    // tuning knobs (environment: PC_QUERY_KERNEL, PC_SORT_BITS), see DESIGN.md §4.6
    int query_kernel = 3;     // packets of ordered batches: 3 = 32 queries, 4 = 64 queries (two per lane)
    bool query_kernel_auto = true;   // PC_QUERY_KERNEL neither 3 nor 4: 3, or 4 for dense batches
    int sort_bits = 24;       // radix-sorted key width of the batch ordering pass (0 = never order)
    bool sort_bits_auto = true;   // no PC_SORT_BITS in the environment: pick 24 or 32 from the batch density
    int next_lane = 0;        // PC_HOST_ASYNC: lane of the next batch
    int shard_rank = 0, shard_n = 1;   // pc_batch_shard
    int key_ctas_per_sm_shard = 0, sortkey_ctas_per_sm_shard = 0;   // occupancy of the pc_batch_shard variants of the key kernels
    float packet_split = 8.f;          // unbounded packet walks: queries farther than this many packet extents from the first one walk separately (PC_PACKET_SPLIT, 0 = off)
    double trace_slow_ms = 0.0;        // PC_TRACE_SLOW_MS: pc_range_batch calls slower than this report their host-side phases
    bool shard_exact = true;           // pc_batch_shard: read the size of the share back (8 bytes, one stream sync) and size the sort / search launches by it
    int radius_arith = PC_ARITH_FP64;  // pc_index_set_radius_arith
    bool onesweep = true;              // PC_ONESWEEP=0: the three-kernel-per-pass radix sort (radix_sort.cuh)
    uint16_t *hilbert_lut = nullptr;   // 16^3 + 32^3 Hilbert indices for the cell binning (pc_hilbert_lut_kernel)
    int key_ctas_per_sm = 0, sortkey_ctas_per_sm = 0;   // occupancy of the bin-count / key kernels (queried once)
    int bin_bits = 0;                  // PC_BIN_BITS: log2 of the number of cells of the binning (0 = from the batch size)
    int coop_group = 0;                     // lanes per query of the small-batch kernel: 0 = by batch size, else 32 / 16 / 8 (PC_COOP_GROUP)
    int64_t coop_g32_max = 6144, coop_g16_max = 12288;   // batch sizes up to which 32 / 16 lanes per query are used (8 above)
    int64_t coop_max = PC_COOP_MAX_BATCH;   // unordered batches up to this size run a group of lanes per query (PC_COOP_MAX_BATCH)
    int64_t coop_max_unbounded = PC_COOP_MAX_BATCH_UNBOUNDED;   // ... unbounded searches (nearest, PC_RADIUS_FULL_NN): their walks are long, and
                                            // beyond 8 k queries one thread per query wins (profiles/r2_coop_group_ab.txt: 24 k nearest 0.17 -> 0.11 ms)
    int64_t sort_min_radius = PC_SORT_MIN_RADIUS, sort_min_nearest = PC_SORT_MIN_NEAREST;   // PC_SORT_MIN_BATCH sets both
    int64_t tiny_batch = PC_TINY_BATCH;   // PC_HOST calls up to this many queries take the mapped-memory path (PC_TINY_BATCH_QUERIES, 0 = off)
    int64_t host_chunk = PC_HOST_CHUNK;   // PC_HOST calls: queries per pipelined chunk (PC_HOST_CHUNK_QUERIES)
    int64_t knn_sort_min = 0;             // pc_knn_batch, PC_QUERY_AUTO: smallest batch that is ordered (PC_KNN_SORT_MIN_BATCH; 0 = by k, knn_host.inl)
    char err[256] = "";
};

// ---- error helpers ---------------------------------------------------------------------------------
static int pc_fail(pc_index *ix, int code, const char *fmt, ...)
{
    char *dst = ix ? ix->err : g_create_error;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(dst, 256, fmt, ap);
    va_end(ap);
    return code;
}

#define PC_CUDA(ix, call)                                                                            \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return pc_fail((ix), e_ == cudaErrorMemoryAllocation ? PC_ENOMEM : PC_ECUDA, "%s: %s", #call, \
                           cudaGetErrorString(e_));                                                  \
    } while (0)

#define PC_CHECK_LAUNCH(ix) PC_CUDA(ix, cudaGetLastError())

// ---- per-call buffers come from the device's stream-ordered memory pool ----------------------------------------------
// A plain cudaMalloc is not a cheap call: on the pool's (virtualised) B200 boxes it stalls the host for 60 - 570 ms every few
// dozen calls (PC_TRACE_SLOW_MS found it in the planner's rewire batches, whose lists grow while the tree grows: 3 of 8 runs
// lost half a second to one allocation).  The buffers that grow with the calls are therefore taken from the default memory
// pool of the device (cudaMallocAsync), which is told never to give memory back to the driver and is warmed at the first
// pc_index_create: once the pool holds the working set, growing a buffer is bookkeeping in user space.  The cloud arena
// (sized by max_points at pc_index_create) stays a plain allocation.
#define PC_POOL_WARM_BYTES ((size_t)256 << 20)      // PC_POOL_WARM_MB overrides

static void pc_pool_setup(int device)
{
    static bool done[64] = { false };
    if (device < 0 || device >= 64 || done[device]) return;
    done[device] = true;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) != cudaSuccess) { cudaGetLastError(); return; }
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    size_t warm = PC_POOL_WARM_BYTES;
    if (const char *v = getenv("PC_POOL_WARM_MB")) { long long b_ = atoll(v); warm = b_ > 0 ? (size_t)b_ << 20 : 0; }
    void *p = nullptr;
    if (warm && cudaMallocAsync(&p, warm, (cudaStream_t)0) == cudaSuccess) { cudaFreeAsync(p, (cudaStream_t)0); cudaStreamSynchronize((cudaStream_t)0); }
    cudaGetLastError();
}

// allocation usable on every stream of the handle when the call returns
static cudaError_t pc_pool_alloc(pc_index *ix, void **p, size_t bytes)
{
    cudaError_t e = cudaMallocAsync(p, bytes, ix->stream);
    if (e != cudaSuccess) { *p = nullptr; return e; }
    return cudaStreamSynchronize(ix->stream);
}

// like cudaFree: nothing on the device may still use the buffer afterwards, whatever stream it ran on
static void pc_pool_free(pc_index *ix, void *p)
{
    if (!p) return;
    cudaDeviceSynchronize();
    cudaFreeAsync(p, ix->stream);
}

template <typename T>
static int pc_grow(pc_index *ix, T **ptr, int64_t *cap, int64_t want, int64_t min_cap = 0)
{
    if (want <= *cap) return PC_OK;
    // buffers never grow by less than a factor of two and never start below 64 Ki elements: a handle reaches its working size
    // within a few calls
    int64_t c = want > min_cap ? want : min_cap;
    if (c < 2 * *cap) c = 2 * *cap;
    if (c < (1 << 16)) c = 1 << 16;
    if (*ptr) { pc_pool_free(ix, *ptr); *ptr = nullptr; *cap = 0; }
    if (pc_pool_alloc(ix, (void **)ptr, (size_t)c * sizeof(T)) != cudaSuccess) {
        cudaGetLastError();                     // no room for the head-room: exactly what was asked for
        c = want > min_cap ? want : min_cap;
        PC_CUDA(ix, pc_pool_alloc(ix, (void **)ptr, (size_t)c * sizeof(T)));
    }
    *cap = c;
    return PC_OK;
}

// the lane's sort buffers (two key and two value buffers of 32-bit words): exactly `want` entries each when they have to grow
static int pc_grow_sort(pc_index *ix, pc_lane &L, int64_t want)
{
    if (want <= L.sort_cap) return PC_OK;
    pc_pool_free(ix, L.keys_a); pc_pool_free(ix, L.keys_b); pc_pool_free(ix, L.vals_a); pc_pool_free(ix, L.vals_b);
    L.keys_a = L.keys_b = L.vals_a = L.vals_b = nullptr; L.sort_cap = 0;
    PC_CUDA(ix, pc_pool_alloc(ix, (void **)&L.keys_a, (size_t)want * 4));
    PC_CUDA(ix, pc_pool_alloc(ix, (void **)&L.keys_b, (size_t)want * 4));
    PC_CUDA(ix, pc_pool_alloc(ix, (void **)&L.vals_a, (size_t)want * 4));
    PC_CUDA(ix, pc_pool_alloc(ix, (void **)&L.vals_b, (size_t)want * 4));
    L.sort_cap = want;
    return PC_OK;
}

static inline int64_t pc_align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// a host array bound for the device (pc_stage_upload)
struct pc_up { const void *src; int64_t bytes; };

// Copy a[0 .. n) to consecutive 256-byte-aligned slots of the device block at dst, on the handle's stream: with `pinned` (the
// slots fit PC_STAGE_BYTES) through the pinned block ix->h_stage in one copy, else one pageable copy per array.  A pageable copy
// costs ~10 us, so the planner's small calls pay for one copy instead of several.
static int pc_stage_upload(pc_index *ix, char *dst, const pc_up *a, int n, bool pinned)
{
    if (pinned && !ix->h_stage) PC_CUDA(ix, cudaHostAlloc((void **)&ix->h_stage, 2 * PC_STAGE_BYTES, cudaHostAllocDefault));
    int64_t o = 0;
    for (int i = 0; i < n; o += pc_align_up(a[i].bytes, 256), i++) {
        if (!pinned) PC_CUDA(ix, cudaMemcpyAsync(dst + o, a[i].src, (size_t)a[i].bytes, cudaMemcpyHostToDevice, ix->stream));
        else if (a[i].bytes > 0) memcpy(ix->h_stage + o, a[i].src, (size_t)a[i].bytes);
    }
    if (pinned) PC_CUDA(ix, cudaMemcpyAsync(dst, ix->h_stage, (size_t)o, cudaMemcpyHostToDevice, ix->stream));
    return PC_OK;
}

// scratch words a sort of n pairs needs: the three-kernel path's tile histograms or the onesweep path's tickets + digit
// histograms + per-pass tile status, whichever is larger
static int64_t pc_sort_scratch_words(int64_t n, int items, int passes)
{
    const int64_t tiles = (n + (int64_t)RS_THREADS * items - 1) / ((int64_t)RS_THREADS * items);
    const int64_t a = (int64_t)RS_RADIX * (tiles + 1), b = os_scratch_words(tiles, passes);
    return a > b ? a : b;
}

// one sort front end: onesweep unless switched off (PC_ONESWEEP=0) or the status words would overflow
template <typename KeyT, int ITEMS>
static int pc_sort_pairs(pc_index *ix, KeyT *keys_a, uint32_t *vals_a, KeyT *keys_b, uint32_t *vals_b, int64_t n, int begin_bit, int end_bit,
                         uint32_t *scratch, uint32_t *digit_total, cudaStream_t st, const unsigned long long *n_dev = nullptr,
                         bool hist_done = false);

static int pc_key_bits_per_axis(int64_t n)
{
    // 10 bits per axis (30-bit keys, 4 radix passes) up to 4 Mi points; beyond that one more bit per axis for
    // every 4x points so that leaves stay spatially tight (surface-like clouds fill ~4^b cells)
    int b = 10;
    int64_t lim = (int64_t)1 << 22;
    while (n > lim && b < 21) { b++; lim <<= 2; }
    return b;
}

// ---- lifetime ----------------------------------------------------------------------------------------
static int pc_reserve_cloud(pc_index *ix, int64_t n)
{
    if (n <= ix->cap) return PC_OK;
    int64_t cap = n;
    // free the old arena
    cudaFree(ix->d_xyz); cudaFree(ix->keys_a); cudaFree(ix->keys_b); cudaFree(ix->vals_a); cudaFree(ix->vals_b);
    cudaFree(ix->tree); cudaFree(ix->tile_hist);
    ix->tree = nullptr; ix->tree_cap = 0;
    ix->d_xyz = nullptr; ix->keys_a = ix->keys_b = nullptr; ix->vals_a = ix->vals_b = nullptr;
    ix->points = nullptr; ix->tile_hist = nullptr; ix->cap = 0; ix->hist_cap = 0;
    ix->key_bytes = pc_key_bits_per_axis(cap) > 10 ? 8 : 4;
    PC_CUDA(ix, cudaMalloc((void **)&ix->d_xyz, (size_t)cap * 4 * sizeof(float)));
    PC_CUDA(ix, cudaMalloc(&ix->keys_a, (size_t)cap * ix->key_bytes));
    PC_CUDA(ix, cudaMalloc(&ix->keys_b, (size_t)cap * ix->key_bytes));
    PC_CUDA(ix, cudaMalloc((void **)&ix->vals_a, (size_t)cap * sizeof(uint32_t)));
    PC_CUDA(ix, cudaMalloc((void **)&ix->vals_b, (size_t)cap * sizeof(uint32_t)));
    ix->tree_cap = 4 * cap + cap + 2 * PC_LEAF + PC_SEED_WORDS / 4 + 1;     // one 64-byte record and one point per point, pad points, seeds
    PC_CUDA(ix, cudaMalloc((void **)&ix->tree, (size_t)ix->tree_cap * sizeof(float4)));
    ix->hist_cap = pc_sort_scratch_words(cap, 8, ix->key_bytes == 8 ? 8 : 4);
    PC_CUDA(ix, cudaMalloc((void **)&ix->tile_hist, (size_t)ix->hist_cap * sizeof(uint32_t)));
    ix->cap = cap;
    return PC_OK;
}

extern "C" int pc_index_create(pc_index **out, int device, int64_t max_points, void *cuda_stream)
{
    if (!out || max_points < 0 || max_points > ((int64_t)1 << 31) - 16) return pc_fail(nullptr, PC_EINVAL, "pc_index_create: bad argument");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return pc_fail(nullptr, PC_ECUDA, "pc_index_create: no CUDA device (%s) -- libpcindex has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return pc_fail(nullptr, PC_EINVAL, "pc_index_create: device %d of %d", device, ndev);
    pc_index *ix = new (std::nothrow) pc_index();
    if (!ix) return pc_fail(nullptr, PC_ENOMEM, "pc_index_create: host allocation failed");
    ix->device = device;
    int rc = PC_OK;
    do {
#define TRY(call) if ((e = (call)) != cudaSuccess) { rc = pc_fail(nullptr, e == cudaErrorMemoryAllocation ? PC_ENOMEM : PC_ECUDA, "%s: %s", #call, cudaGetErrorString(e)); break; }
        TRY(cudaSetDevice(device));
        pc_pool_setup(device);
        cudaDeviceProp prop;
        TRY(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10) { rc = pc_fail(nullptr, PC_ECUDA, "pc_index_create: device is sm_%d%d, this library is built for sm_100a only", prop.major, prop.minor); break; }
        ix->sm_count = prop.multiProcessorCount;
        // PC_QUERY_KERNEL: 3 or 4 forces 32- or 64-query packets; any other value is ignored (the batch density decides)
        if (const char *v = getenv("PC_QUERY_KERNEL")) { int b_ = atoi(v); if (b_ == 3 || b_ == 4) { ix->query_kernel_auto = false; ix->query_kernel = b_; } }
        if (const char *v = getenv("PC_SORT_BITS")) { ix->sort_bits_auto = false; int b_ = atoi(v); ix->sort_bits = b_ <= 0 ? 0 : (b_ <= 16 ? 16 : (b_ <= 24 ? 24 : 32)); }
        if (const char *v = getenv("PC_ONESWEEP")) ix->onesweep = atoi(v) != 0;
        if (const char *v = getenv("PC_BIN_BITS")) { int b_ = atoi(v); ix->bin_bits = b_ < 12 ? 0 : (b_ > PC_BIN_MAX_BITS ? PC_BIN_MAX_BITS : b_); }
        if (const char *v = getenv("PC_SHARD_EXACT")) ix->shard_exact = atoi(v) != 0;
        if (const char *v = getenv("PC_TRACE_SLOW_MS")) ix->trace_slow_ms = atof(v);
        if (const char *v = getenv("PC_PACKET_SPLIT")) { double c_ = atof(v); ix->packet_split = c_ > 0.0 ? (float)c_ : 0.f; }
        if (const char *v = getenv("PC_HOST_CHUNK_QUERIES")) { long long b_ = atoll(v); if (b_ >= 1024) ix->host_chunk = b_; }
        if (const char *v = getenv("PC_COOP_GROUP")) { int b_ = atoi(v); ix->coop_group = (b_ == 32 || b_ == 16 || b_ == 8) ? b_ : 0; }
        if (const char *v = getenv("PC_COOP_MAX_BATCH")) { long long b_ = atoll(v); ix->coop_max = ix->coop_max_unbounded = b_ < 0 ? 0 : b_; }
        if (const char *v = getenv("PC_SORT_MIN_BATCH")) { long long b_ = atoll(v); ix->sort_min_radius = ix->sort_min_nearest = b_ < 1 ? 1 : b_; }
        if (const char *v = getenv("PC_KNN_SORT_MIN_BATCH")) { long long b_ = atoll(v); ix->knn_sort_min = b_ < 0 ? 0 : b_; }
        if (const char *v = getenv("PC_TINY_BATCH_QUERIES")) { long long b_ = atoll(v); ix->tiny_batch = b_ < 0 ? 0 : (b_ > PC_TINY_BATCH ? PC_TINY_BATCH : b_); }
        if (cuda_stream) { ix->stream = (cudaStream_t)cuda_stream; ix->own_stream = false; }
        else { TRY(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking)); ix->own_stream = true; }
        TRY(cudaEventCreate(&ix->ev_b0));
        TRY(cudaEventCreate(&ix->ev_b1));
        TRY(cudaEventCreateWithFlags(&ix->ev_ready, cudaEventDisableTiming));
        TRY(cudaEventCreateWithFlags(&ix->ev_in, cudaEventDisableTiming));
        TRY(cudaMalloc((void **)&ix->d_bbox, 8 * sizeof(uint32_t)));
        TRY(cudaHostAlloc((void **)&ix->h_bbox, 8 * sizeof(uint32_t), cudaHostAllocDefault));
        TRY(cudaMalloc((void **)&ix->digit_total, RS_RADIX * sizeof(uint32_t)));
        // the Hilbert lookup tables of the cell binning: filled here, once, so that every stream of the handle may read them
        TRY(cudaMalloc((void **)&ix->hilbert_lut, (size_t)(PC_LUT4_WORDS + PC_LUT5_WORDS) * sizeof(uint16_t)));
        pc_hilbert_lut_kernel<<<PC_LUT5_WORDS / 256, 256, 0, ix->stream>>>(ix->hilbert_lut, ix->hilbert_lut + PC_LUT4_WORDS);
        TRY(cudaGetLastError());
        TRY(cudaStreamSynchronize(ix->stream));
        TRY(cudaHostAlloc((void **)&ix->tiny_q, PC_TINY_BATCH * 4 * sizeof(float), cudaHostAllocMapped));
        TRY(cudaHostAlloc((void **)&ix->tiny_f, PC_TINY_BATCH * sizeof(float), cudaHostAllocMapped));
        TRY(cudaHostAlloc((void **)&ix->tiny_i, PC_TINY_BATCH * sizeof(int32_t), cudaHostAllocMapped));
        TRY(cudaHostGetDevicePointer((void **)&ix->tiny_q_dev, ix->tiny_q, 0));
        TRY(cudaHostGetDevicePointer((void **)&ix->tiny_f_dev, ix->tiny_f, 0));
        TRY(cudaHostGetDevicePointer((void **)&ix->tiny_i_dev, ix->tiny_i, 0));
        for (int l = 0; l < PC_PIPE_LANES; l++) {
            // lane 0 shares the handle's stream (PC_DEVICE calls are ordered on it); the others overlap copies
            if (l == 0) { ix->lane[l].stream = ix->stream; ix->lane[l].own_stream = false; }
            else { TRY(cudaStreamCreateWithFlags(&ix->lane[l].stream, cudaStreamNonBlocking)); ix->lane[l].own_stream = true; }
            TRY(cudaEventCreateWithFlags(&ix->lane[l].done, cudaEventDisableTiming));
            TRY(cudaEventCreateWithFlags(&ix->lane[l].ev_deps, cudaEventDisableTiming));
            TRY(cudaEventCreateWithFlags(&ix->lane[l].ev_ordered, cudaEventDisableTiming));
            {
                int lo_p = 0, hi_p = 0;
                TRY(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
                TRY(cudaStreamCreateWithPriority(&ix->lane[l].order_stream, cudaStreamNonBlocking, hi_p));
            }
            TRY(cudaEventCreate(&ix->lane[l].t0));
            TRY(cudaEventCreate(&ix->lane[l].t1));
            TRY(cudaEventCreate(&ix->lane[l].t2));
            TRY(cudaEventCreate(&ix->lane[l].ta));
            TRY(cudaEventCreate(&ix->lane[l].tb));
            TRY(cudaMalloc((void **)&ix->lane[l].digit_total, RS_RADIX * sizeof(uint32_t)));
            TRY(cudaMalloc((void **)&ix->lane[l].counter, 2 * sizeof(unsigned long long)));
        }
        if (rc != PC_OK) break;
#undef TRY
        if (max_points > 0) {
            rc = pc_reserve_cloud(ix, max_points);
            if (rc != PC_OK) { strncpy(g_create_error, ix->err, 255); break; }
        }
    } while (0);
    if (rc != PC_OK) { pc_index_destroy(ix); return rc; }
    *out = ix;
    return PC_OK;
}

extern "C" void pc_index_destroy(pc_index *ix)
{
    if (!ix) return;
    cudaSetDevice(ix->device);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    for (int l = 0; l < PC_PIPE_LANES; l++) {
        pc_lane &L = ix->lane[l];
        if (L.stream && L.own_stream) { cudaStreamSynchronize(L.stream); cudaStreamDestroy(L.stream); }
        cudaFree(L.d_q); cudaFree(L.d_i32); cudaFree(L.d_f32);
        cudaFree(L.keys_a); cudaFree(L.keys_b); cudaFree(L.vals_a); cudaFree(L.vals_b);
        cudaFree(L.tile_hist); cudaFree(L.digit_total); cudaFree(L.counter); cudaFree(L.bins); cudaFree(L.ordered); cudaFree(L.d_mid);
        if (L.done) cudaEventDestroy(L.done);
        if (L.ev_deps) cudaEventDestroy(L.ev_deps);
        if (L.ev_ordered) cudaEventDestroy(L.ev_ordered);
        if (L.order_stream) { cudaStreamSynchronize(L.order_stream); cudaStreamDestroy(L.order_stream); }
        if (L.t0) cudaEventDestroy(L.t0);
        if (L.t1) cudaEventDestroy(L.t1);
        if (L.t2) cudaEventDestroy(L.t2);
        if (L.ta) cudaEventDestroy(L.ta);
        if (L.tb) cudaEventDestroy(L.tb);
    }
    if (ix->h_bbox) cudaFreeHost(ix->h_bbox);
    if (ix->h_totals) cudaFreeHost(ix->h_totals);
    if (ix->h_stage) cudaFreeHost(ix->h_stage);
    for (int i = 0; i < 2; i++) if (ix->ev_chunk[i]) cudaEventDestroy(ix->ev_chunk[i]);
    if (ix->tiny_q) cudaFreeHost(ix->tiny_q);
    if (ix->tiny_f) cudaFreeHost(ix->tiny_f);
    if (ix->tiny_i) cudaFreeHost(ix->tiny_i);
    cudaFree(ix->d_xyz); cudaFree(ix->d_bbox); cudaFree(ix->keys_a); cudaFree(ix->keys_b);
    cudaFree(ix->vals_a); cudaFree(ix->vals_b); cudaFree(ix->tile_hist); cudaFree(ix->digit_total);
    cudaFree(ix->tree); cudaFree(ix->scratch); cudaFree(ix->range_long); cudaFree(ix->hilbert_lut);
    if (ix->ev_b0) cudaEventDestroy(ix->ev_b0);
    if (ix->ev_b1) cudaEventDestroy(ix->ev_b1);
    if (ix->ev_ready) cudaEventDestroy(ix->ev_ready);
    if (ix->ev_in) cudaEventDestroy(ix->ev_in);
    if (ix->own_stream && ix->stream) cudaStreamDestroy(ix->stream);
    delete ix;
}

extern "C" int pc_index_sync(pc_index *ix)
{
    if (!ix) return PC_EINVAL;
    PC_CUDA(ix, cudaSetDevice(ix->device));
    PC_CUDA(ix, cudaStreamSynchronize(ix->stream));
    for (int l = 1; l < PC_PIPE_LANES; l++) PC_CUDA(ix, cudaStreamSynchronize(ix->lane[l].stream));   // PC_HOST_ASYNC batches
    return PC_OK;
}

extern "C" const char *pc_last_error(const pc_index *ix) { return ix ? ix->err : g_create_error; }
extern "C" const char *pc_version(void) { return PC_VERSION_STRING; }
extern "C" int64_t pc_index_size(const pc_index *ix) { return ix ? ix->n : 0; }

extern "C" int64_t pc_launch_count(const pc_index *ix, int reset)
{
    if (!ix) return 0;
    int64_t v = ix->launches;
    if (reset) const_cast<pc_index *>(ix)->launches = 0;
    return v;
}

extern "C" void *pc_host_alloc(int64_t bytes)
{
    void *p = nullptr;
    if (bytes <= 0) return nullptr;
    if (cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}

extern "C" void pc_host_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" void pc_shard_range(int64_t m, int rank, int n_ranks, int64_t *begin, int64_t *end)
{
    if (n_ranks < 1) n_ranks = 1;
    if (rank < 0) rank = 0;
    if (rank >= n_ranks) rank = n_ranks - 1;
    int64_t base = m / n_ranks, rem = m % n_ranks;
    int64_t b = rank * base + (rank < rem ? rank : rem);
    int64_t e = b + base + (rank < rem ? 1 : 0);
    if (begin) *begin = b;
    if (end) *end = e;
}

// ---- index build -----------------------------------------------------------------------------------
template <typename KeyT, int ITEMS>
static int pc_build_sorted(pc_index *ix, const float *src, int stride, int64_t n, int bits, uint32_t **order_out, void **keys_out)
{
    cudaStream_t st = ix->stream;
    const int grid = (int)((n + PC_BUILD_THREADS - 1) / PC_BUILD_THREADS < (int64_t)ix->sm_count * 8
                               ? (n + PC_BUILD_THREADS - 1) / PC_BUILD_THREADS : (int64_t)ix->sm_count * 8);
    int key_bits = 3 * bits;
    int end_bit = ((key_bits + 7) / 8) * 8;
    const bool fused_hist = ix->onesweep && n < OS_MAX_N;      // the key kernel also counts the sort's digit histograms
    if (fused_hist) os_clear(ix->tile_hist, n, ITEMS, end_bit / 8, st);
    pc_keygen_kernel<KeyT><<<grid, PC_BUILD_THREADS, 0, st>>>(src, n, stride, ix->d_bbox, bits, (KeyT *)ix->keys_a, ix->vals_a,
                                                              fused_hist ? os_ghist(ix->tile_hist) : nullptr, end_bit / 8);
    ix->launches++;
    PC_CHECK_LAUNCH(ix);
    int which = pc_sort_pairs<KeyT, ITEMS>(ix, (KeyT *)ix->keys_a, ix->vals_a, (KeyT *)ix->keys_b, ix->vals_b, n, 0, end_bit,
                                           ix->tile_hist, ix->digit_total, st, nullptr, fused_hist);
    PC_CHECK_LAUNCH(ix);
    *order_out = which ? ix->vals_b : ix->vals_a;
    *keys_out = which ? ix->keys_b : ix->keys_a;
    return PC_OK;
}

extern "C" int pc_index_build(pc_index *ix, const float *xyz, int64_t n, int64_t stride_floats, int space)
{
    if (!ix) return PC_EINVAL;
    if (n < 0 || (n > 0 && !xyz) || (stride_floats != 3 && stride_floats != 4) || (space != PC_HOST && space != PC_DEVICE))
        return pc_fail(ix, PC_EINVAL, "pc_index_build: bad argument (n=%lld stride=%lld space=%d)", (long long)n, (long long)stride_floats, space);
    if (n > ((int64_t)1 << 31) - 16) return pc_fail(ix, PC_EINVAL, "pc_index_build: at most 2^31-16 points");
    PC_CUDA(ix, cudaSetDevice(ix->device));
    if (n == 0) { ix->n = 0; ix->n_nodes = 0; ix->root = PC_REF_LEAF; ix->root_count = 0; ix->build_timed = false; return PC_OK; }
    if (n > ix->cap) {
        PC_CUDA(ix, cudaStreamSynchronize(ix->stream));
        int rc = pc_reserve_cloud(ix, n);
        if (rc != PC_OK) return rc;
    }
    cudaStream_t st = ix->stream;
    // batches still in flight on the side lanes (PC_HOST_ASYNC) read the tree this build is about to overwrite
    for (int l = 1; l < PC_PIPE_LANES; l++) PC_CUDA(ix, cudaStreamWaitEvent(st, ix->lane[l].done, 0));
    const int stride = (int)stride_floats;
    const float *src = xyz;
    if (space == PC_HOST) {
        PC_CUDA(ix, cudaMemcpyAsync(ix->d_xyz, xyz, (size_t)n * stride * sizeof(float), cudaMemcpyHostToDevice, st));
        src = ix->d_xyz;
    }
    PC_CUDA(ix, cudaEventRecord(ix->ev_b0, st));
    // bbox: [0..2] = 0xffffffff (ordered +max) for the minima, [3..5] = 0 for the maxima
    PC_CUDA(ix, cudaMemsetAsync(ix->d_bbox, 0xff, 3 * sizeof(uint32_t), st));
    PC_CUDA(ix, cudaMemsetAsync(ix->d_bbox + 3, 0x00, 3 * sizeof(uint32_t), st));
    {
        int64_t blocks = (n + PC_BUILD_THREADS - 1) / PC_BUILD_THREADS;
        int grid = (int)(blocks < (int64_t)ix->sm_count * 4 ? blocks : (int64_t)ix->sm_count * 4);
        pc_bbox_kernel<<<grid, PC_BUILD_THREADS, 0, st>>>(src, n, stride, ix->d_bbox);
        ix->launches++;
        PC_CHECK_LAUNCH(ix);
    }
    const int bits = pc_key_bits_per_axis(n);
    uint32_t *order = nullptr;
    void *sorted_keys = nullptr;
    int rc;
    const bool big = n > ((int64_t)1 << 21);
    if (bits <= 10) {
        if (ix->key_bytes < 4) return pc_fail(ix, PC_ECUDA, "internal: key buffer");
        rc = big ? pc_build_sorted<uint32_t, 16>(ix, src, stride, n, bits, &order, &sorted_keys)
                 : pc_build_sorted<uint32_t, 8>(ix, src, stride, n, bits, &order, &sorted_keys);
    } else {
        if (ix->key_bytes < 8) return pc_fail(ix, PC_ECUDA, "internal: key buffer too narrow");
        rc = pc_build_sorted<uint64_t, 8>(ix, src, stride, n, bits, &order, &sorted_keys);
    }
    if (rc != PC_OK) return rc;

    // the radix tree over the sorted keys: records [0, 4 (n-1)), then the points in curve order.  The sort's spare buffers
    // (the ones that do NOT hold the sorted result) serve as parent links and arrival counters of the bottom-up fit.
    const int64_t n_nodes = n > PC_LEAF ? n - 1 : 0;
    ix->points = ix->tree + 4 * n_nodes;
    {
        int32_t *parent = (int32_t *)(order == ix->vals_a ? ix->vals_b : ix->vals_a);
        int *arrived = (int *)(sorted_keys == ix->keys_a ? ix->keys_b : ix->keys_a);
        const int grid = (int)((n + PC_LEAF + PC_BUILD_THREADS - 1) / PC_BUILD_THREADS);
        if (bits <= 10)
            pc_tree_nodes_kernel<uint32_t><<<grid, PC_BUILD_THREADS, 0, st>>>(src, stride, order, (const uint32_t *)sorted_keys, n, ix->tree, ix->points, parent, arrived);
        else
            pc_tree_nodes_kernel<uint64_t><<<grid, PC_BUILD_THREADS, 0, st>>>(src, stride, order, (const uint64_t *)sorted_keys, n, ix->tree, ix->points, parent, arrived);
        ix->launches++;
        PC_CHECK_LAUNCH(ix);
        if (n_nodes > 0) {
            pc_tree_fit_kernel<<<(int)((n_nodes + PC_BUILD_THREADS - 1) / PC_BUILD_THREADS), PC_BUILD_THREADS, 0, st>>>(ix->tree, ix->points, parent, arrived, n);
            ix->launches++;
            PC_CHECK_LAUNCH(ix);
        }
        // the seeds of the lane-group walks sit right behind the points (the records' child references are final after the
        // nodes kernel; the boxes are not needed)
        pc_tree_seed_kernel<<<1, 32, 0, st>>>(ix->tree, n_nodes > 0 ? 0u : PC_REF_LEAF, n_nodes > 0 ? 0u : (uint32_t)n,
                                               reinterpret_cast<uint32_t *>(ix->points + n + PC_LEAF));
        ix->launches++;
        PC_CHECK_LAUNCH(ix);
    }
    PC_CUDA(ix, cudaMemcpyAsync(ix->h_bbox, ix->d_bbox, 6 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PC_CUDA(ix, cudaEventRecord(ix->ev_b1, st));
    PC_CUDA(ix, cudaEventRecord(ix->ev_ready, st));
    ix->n = n; ix->n_nodes = n_nodes; ix->build_timed = true; ix->bbox_from_bcast = false;
    ix->root = n_nodes > 0 ? 0u : PC_REF_LEAF; ix->root_count = n_nodes > 0 ? 0u : (uint32_t)n;
    if (space == PC_HOST) PC_CUDA(ix, cudaStreamSynchronize(st));
    return PC_OK;
}

template <typename KeyT, int ITEMS>
static int pc_sort_pairs(pc_index *ix, KeyT *keys_a, uint32_t *vals_a, KeyT *keys_b, uint32_t *vals_b, int64_t n, int begin_bit, int end_bit,
                         uint32_t *scratch, uint32_t *digit_total, cudaStream_t st, const unsigned long long *n_dev, bool hist_done)
{
    if (ix->onesweep && n < OS_MAX_N)
        return os_sort_pairs<KeyT, ITEMS>(keys_a, vals_a, keys_b, vals_b, n, begin_bit, end_bit, scratch, ix->sm_count, st, &ix->launches, n_dev, hist_done);
    return rs_sort_pairs<KeyT, ITEMS>(keys_a, vals_a, keys_b, vals_b, n, begin_bit, end_bit, scratch, digit_total, st, &ix->launches, n_dev);
}

extern "C" int pc_index_last_build_ms(pc_index *ix, float *ms)
{
    if (!ix || !ms) return PC_EINVAL;
    if (!ix->build_timed) { *ms = 0.f; return PC_OK; }
    PC_CUDA(ix, cudaSetDevice(ix->device));
    PC_CUDA(ix, cudaEventSynchronize(ix->ev_b1));
    PC_CUDA(ix, cudaEventElapsedTime(ms, ix->ev_b0, ix->ev_b1));
    return PC_OK;
}

extern "C" int pc_index_view_get(const pc_index *ixc, pc_index_view *out)
{
    pc_index *ix = const_cast<pc_index *>(ixc);
    if (!ix || !out) return PC_EINVAL;
    memset(out, 0, sizeof *out);
    out->n_points = ix->n; out->n_nodes = ix->n_nodes; out->root = ix->root; out->root_count = ix->root_count;
    out->points = ix->points; out->records = ix->tree;
    if (ix->n > 0) {
        uint32_t h[6];
        PC_CUDA(ix, cudaSetDevice(ix->device));
        PC_CUDA(ix, cudaMemcpyAsync(h, ix->d_bbox, sizeof h, cudaMemcpyDeviceToHost, ix->stream));
        PC_CUDA(ix, cudaStreamSynchronize(ix->stream));
        for (int a = 0; a < 3; a++) { out->bbox_lo[a] = pc_ordered_to_float(h[a]); out->bbox_hi[a] = pc_ordered_to_float(h[3 + a]); }
    }
    return PC_OK;
}

// ---- query plumbing ----------------------------------------------------------------------------------
static pc_tree pc_tree_of(const pc_index *ix)
{
    pc_tree T;
    T.rec = ix->tree; T.points = ix->points; T.n_points = ix->n; T.root = ix->root; T.root_count = ix->root_count;
    T.seeds = reinterpret_cast<const uint32_t *>(ix->points + ix->n + PC_LEAF);
    return T;
}

enum pc_qkind { PC_Q_NEAREST, PC_Q_RADIUS };

struct pc_qargs {
    pc_qkind kind;
    pc_radius_dev R;
    int flags;
};

static pc_qargs pc_nearest_qargs(int flags)
{
    pc_qargs A;
    memset(&A, 0, sizeof A);
    A.kind = PC_Q_NEAREST; A.flags = flags;
    return A;
}

// pc_batch_shard: the number of queries of this rank's share (L.counter[1], written by the ordering kernels queued on L.os)
static int pc_share_size(pc_index *ix, pc_lane &L, int64_t m, int64_t *out)
{
    unsigned long long h = 0;
    PC_CUDA(ix, cudaMemcpyAsync(&h, L.counter + 1, sizeof h, cudaMemcpyDeviceToHost, L.os));
    PC_CUDA(ix, cudaStreamSynchronize(L.os));
    *out = (int64_t)h < m ? (int64_t)h : m;
    return PC_OK;
}

// Whether a row-per-query batch of m entries is put in curve order: always on a pc_batch_shard handle (the share is selected
// by the ordering pass), as PC_QUERY_SORTED / PC_QUERY_UNSORTED say, and under PC_QUERY_AUTO from the caller's sort_min on.
static bool pc_want_order(const pc_index *ix, int flags, int64_t m, int64_t sort_min)
{
    if (ix->n == 0 || ix->sort_bits == 0) return false;
    if (ix->shard_n > 1) return true;
    if (flags & PC_QUERY_SORTED) return true;
    if (flags & PC_QUERY_UNSORTED) return false;
    return m >= sort_min;
}

// the smallest nearest / radius batch that PC_QUERY_AUTO orders
static int64_t pc_sort_min(const pc_index *ix, const pc_qargs &A)
{
    return A.kind == PC_Q_NEAREST || !A.R.bounded ? ix->sort_min_nearest : ix->sort_min_radius;
}

// The ordering step of every row-per-query batch (pc_run_batch, the kNN, kNN-large and segment runs) on lane L, queued on
// L.os: when pc_want_order says so, the m entries are put in curve order over the points d_a (stride floats per row), or with
// d_b over the midpoints of the segments [d_a, d_b].  L.counter is zeroed first (counter[0]: the packet walks' deferred
// packets, counter[1]: the entries left to search, written by this pass).  Radius batches (A) answer their sensing-range
// early-outs here, into d_idx / d_f.  A batch left in its own order gets perm = ordered = m_eff = nullptr, m_launch = m.
struct pc_order {
    const uint32_t *perm;
    const float4 *ordered;
    const unsigned long long *m_eff;    // entries to search (written by the ordering pass)
    int64_t m_launch;                   // host-side bound of *m_eff: the launches are sized by it (the exact share in pc_batch_shard mode)
};

static int pc_order_batch(pc_index *ix, pc_lane &L, const pc_qargs &A, int64_t sort_min, const float *d_a, const float *d_b,
                          int64_t m, int stride, int32_t *d_idx, float *d_f, bool may_sync, pc_order &O)
{
    O.perm = nullptr; O.ordered = nullptr; O.m_eff = nullptr; O.m_launch = m;
    if (!pc_want_order(ix, A.flags, m, sort_min)) return PC_OK;
    const float *d_q = d_a;
    int qstride = stride;
    if (d_b) {
        int rcm = pc_grow(ix, &L.d_mid, &L.mid_cap, m);
        if (rcm != PC_OK) return rcm;
        const int64_t blocks = (m + 255) / 256;
        pc_seg_mid_kernel<<<(int)(blocks < ix->sm_count * 8 ? blocks : ix->sm_count * 8), 256, 0, L.os>>>(d_a, d_b, m, stride, L.d_mid);
        ix->launches++;
        d_q = reinterpret_cast<const float *>(L.d_mid);
        qstride = 4;
    }
    PC_CUDA(ix, cudaMemsetAsync(L.counter, 0, 2 * sizeof(unsigned long long), L.os));
    O.m_eff = L.counter + 1;
    // pc_batch_shard: a rank searches about 1 / shard_n of the batch, but how many exactly is known on the device only, and
    // launches sized for the whole batch are mostly CTAs that find nothing to do (C5 on 8 GPUs: 683 k of 781 k search CTAs and
    // 7 of 8 sort tiles; more than a millisecond of an 8 ms call).  Large sharded batches therefore read the count back --
    // 8 bytes and one synchronisation of the ordering stream -- and size every later launch by it.  PC_DEVICE calls only:
    // the pipelined spaces (chunked PC_HOST, the ASYNC ones) must not stall the host between their copies.
    const bool exact = may_sync && ix->shard_n > 1 && ix->shard_exact && m >= PC_SHARD_EXACT_MIN;
    int rc = pc_grow_sort(ix, L, m);
    if (rc != PC_OK) return rc;
    rc = pc_grow(ix, &L.tile_hist, &L.hist_cap, pc_sort_scratch_words(m, 8, 4));
    if (rc != PC_OK) return rc;
    // sort_bits (16 / 24 / 32) = radix-sorted key width = how many of the top curve bits order the batch; queries that
    // need no search (sensing-range early-outs) are answered by the key kernel and never enter the sort
    int bits = ix->sort_bits;
    L.per_cell = 0.0;
    if (ix->sort_bits_auto && ((ix->build_timed && cudaEventQuery(ix->ev_b1) == cudaSuccess) || ix->bbox_from_bcast)) {
        // 24 bits (8 per axis) order the batch well when its cells hold a handful of queries; a batch that is dense
        // relative to the cloud's extent (large maps) needs the full 30-bit curve.  Estimated from the cloud's bounding
        // box; if the build has not finished yet (no host copy of the box) the default stays.
        float ext[3], emax = 0.f, vol = 1.f;
        for (int a = 0; a < 3; a++) {
            ext[a] = pc_ordered_to_float(ix->h_bbox[3 + a]) - pc_ordered_to_float(ix->h_bbox[a]);
            emax = ext[a] > emax ? ext[a] : emax;
        }
        for (int a = 0; a < 3; a++) vol *= ext[a] > emax / 256.f ? ext[a] : emax / 256.f;
        const float cell = emax / 256.f;
        const double per_cell = vol > 0.f ? (double)m * cell * cell * cell / vol : 0.0;
        bits = per_cell > 16.0 ? 32 : 24;
        L.per_cell = per_cell;
    }
    const bool prof = ix->profile && &L == &ix->lane[0];
    // (bounded radius batches only: unbounded nearest batches measured 5 % slower end to end on the binned order -- their
    // search is 11 % slower on it, profiles/r2_order_bins_sweep.txt -- and keep the radix sort)
    if (bits == 24 && m < ((int64_t)1 << 32) - 1 && A.kind == PC_Q_RADIUS && A.R.bounded) {
        // cell binning (query_kernels.cuh): counting sort by the 21-bit Hilbert cell, the queries themselves gathered into
        // cell order.  Taken whenever the density test would have picked the 24-bit radix sort.
        // number of cells: about half the batch size (a handful of queries per occupied cell, like the 24-bit radix order),
        // 2^18 .. 2^24; PC_BIN_BITS overrides
        int bin_bits = ix->bin_bits;
        if (bin_bits == 0) { bin_bits = 17; while (bin_bits < PC_BIN_MAX_BITS && ((int64_t)1 << (bin_bits + 2)) <= m) bin_bits++; }
        const int64_t n_bins = (int64_t)1 << bin_bits;
        int rcb = pc_grow(ix, &L.bins, &L.bins_cap, n_bins + n_bins / PC_BIN_SCAN_TILE + 64);
        if (rcb != PC_OK) return rcb;
        if ((rcb = pc_grow(ix, &L.ordered, &L.ordered_cap, m)) != PC_OK) return rcb;
        if (ix->key_ctas_per_sm == 0) {
            PC_CUDA(ix, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ix->key_ctas_per_sm, pc_bin_count_kernel<false>, 256, 0));
            PC_CUDA(ix, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ix->key_ctas_per_sm_shard, pc_bin_count_kernel<true>, 256, 0));
            if (ix->key_ctas_per_sm_shard < 1) ix->key_ctas_per_sm_shard = 1;
            if (ix->key_ctas_per_sm < 1) ix->key_ctas_per_sm = 1;
        }
        const int64_t rounds = (m + 256 * PC_KEY_ITEMS - 1) / (256 * PC_KEY_ITEMS);
        const bool sharded = ix->shard_n > 1;
        const int64_t wave = (int64_t)ix->sm_count * (sharded ? ix->key_ctas_per_sm_shard : ix->key_ctas_per_sm);
        const int grid = (int)(rounds < wave ? rounds : wave);
        uint32_t *tile_sum = L.bins + n_bins;
        const int n_tiles = (int)(n_bins / PC_BIN_SCAN_TILE);
        PC_CUDA(ix, cudaMemsetAsync(L.bins, 0, (size_t)n_bins * sizeof(uint32_t), L.os));
        if (prof) PC_CUDA(ix, cudaEventRecord(L.ta, L.os));
#define PC_BIN_COUNT(S) pc_bin_count_kernel<S><<<grid, 256, 0, L.os>>>(d_q, m, qstride, ix->d_bbox, A.R, d_idx, d_f, L.keys_a, L.bins, bin_bits, ix->shard_rank, ix->shard_n, ix->hilbert_lut)
        if (sharded) PC_BIN_COUNT(true); else PC_BIN_COUNT(false);
#undef PC_BIN_COUNT
        if (prof) PC_CUDA(ix, cudaEventRecord(L.tb, L.os));
        pc_bin_scan_tiles<<<n_tiles, 256, 0, L.os>>>(L.bins, tile_sum);
        pc_bin_scan_top<<<1, 1024, 0, L.os>>>(tile_sum, n_tiles, L.counter + 1);
        pc_bin_scan_apply<<<n_tiles, 256, 0, L.os>>>(L.bins, tile_sum);
        // (sharded: a query of another rank costs the scatter its 4-byte cell key only)
        if (sharded)
            pc_bin_scatter_kernel<true><<<grid, 256, 0, L.os>>>(d_q, m, qstride, L.keys_a, L.bins, L.ordered);
        else
            pc_bin_scatter_kernel<false><<<grid, 256, 0, L.os>>>(d_q, m, qstride, L.keys_a, L.bins, L.ordered);
        ix->launches += 5;
        PC_CHECK_LAUNCH(ix);
        O.ordered = L.ordered;
        if (exact) return pc_share_size(ix, L, m, &O.m_launch);
        return PC_OK;
    }
    const int drop = 30 - bits > 0 ? 30 - bits : 0;     // 24-bit sort = top 24 curve bits, 32-bit sort = all 30
    // one wave of CTAs (as many as the key kernel's occupancy allows), each striding over the batch
    if (ix->sortkey_ctas_per_sm == 0) {
        int a = 0, b = 0;
        int c = 0, d = 0;
        PC_CUDA(ix, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, pc_query_key_kernel<PC_KIND_RADIUS, false>, 256, 0));
        PC_CUDA(ix, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, pc_query_key_kernel<PC_KIND_NEAREST, false>, 256, 0));
        PC_CUDA(ix, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c, pc_query_key_kernel<PC_KIND_RADIUS, true>, 256, 0));
        PC_CUDA(ix, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&d, pc_query_key_kernel<PC_KIND_NEAREST, true>, 256, 0));
        ix->sortkey_ctas_per_sm = a < b ? a : b;
        if (ix->sortkey_ctas_per_sm < 1) ix->sortkey_ctas_per_sm = 1;
        ix->sortkey_ctas_per_sm_shard = c < d ? c : d;
        if (ix->sortkey_ctas_per_sm_shard < 1) ix->sortkey_ctas_per_sm_shard = 1;
    }
    const bool sharded = ix->shard_n > 1;
    const int64_t key_ctas = (m + 256 * PC_KEY_ITEMS - 1) / (256 * PC_KEY_ITEMS);
    const int64_t key_wave = (int64_t)ix->sm_count * (sharded ? ix->sortkey_ctas_per_sm_shard : ix->sortkey_ctas_per_sm);
    const int grid = (int)(key_ctas < key_wave ? key_ctas : key_wave);
    constexpr int items = 16;          // keys per thread of the ordering sort
    const bool fused_hist = ix->onesweep && m < OS_MAX_N;
    uint32_t *gh = fused_hist ? os_ghist(L.tile_hist) : nullptr;
    if (fused_hist) {
        // (exact share: tickets and digit histograms now, the tile status words once the number of tiles is known)
        if (exact) PC_CUDA(ix, cudaMemsetAsync(L.tile_hist, 0, (size_t)os_scratch_words(0, bits / 8) * sizeof(uint32_t), L.os));
        else os_clear(L.tile_hist, m, items, bits / 8, L.os);
    }
    if (prof) PC_CUDA(ix, cudaEventRecord(L.ta, L.os));
#define PC_QUERY_KEY(K, S) pc_query_key_kernel<K, S><<<grid, 256, 0, L.os>>>(d_q, m, qstride, ix->d_bbox, drop, A.R, d_idx, d_f, L.keys_a, L.vals_a, L.counter + 1, ix->shard_rank, ix->shard_n, gh, bits / 8)
    if (A.kind == PC_Q_RADIUS) { if (sharded) PC_QUERY_KEY(PC_KIND_RADIUS, true); else PC_QUERY_KEY(PC_KIND_RADIUS, false); }
    else { if (sharded) PC_QUERY_KEY(PC_KIND_NEAREST, true); else PC_QUERY_KEY(PC_KIND_NEAREST, false); }
#undef PC_QUERY_KEY
    ix->launches++;
    PC_CHECK_LAUNCH(ix);
    if (prof) PC_CUDA(ix, cudaEventRecord(L.tb, L.os));
    int64_t n_sort = m;
    if (exact) {
        int rcs = pc_share_size(ix, L, m, &n_sort);
        if (rcs != PC_OK) return rcs;
        O.m_launch = n_sort;
        if (n_sort == 0) { O.perm = L.vals_a; return PC_OK; }
        if (fused_hist) {
            const int64_t tiles = (n_sort + (int64_t)RS_THREADS * items - 1) / ((int64_t)RS_THREADS * items);
            PC_CUDA(ix, cudaMemsetAsync(L.tile_hist + os_scratch_words(0, bits / 8), 0, (size_t)(os_scratch_words(tiles, bits / 8) - os_scratch_words(0, bits / 8)) * sizeof(uint32_t), L.os));
        }
    }
    // only the L.counter[1] compacted entries (device-side count <= m; n_sort bounds it on the host) are sorted
    int which = pc_sort_pairs<uint32_t, items>(ix, L.keys_a, L.vals_a, L.keys_b, L.vals_b, n_sort, 0, bits, L.tile_hist, L.digit_total, L.os, L.counter + 1, fused_hist);
    PC_CHECK_LAUNCH(ix);
    O.perm = which ? L.vals_b : L.vals_a;
    return PC_OK;
}

// small unordered batch: G lanes per query.  A whole warp per query has the lowest latency while the batch fits the GPU's
// resident warps; beyond that, narrower groups put more queries in flight (scripts/small_batch_ab.py).
template <int G>
static void pc_launch_coop_g(const pc_qargs &A, const pc_tree &T, const float *d_q, int64_t m, int qstride,
                             int32_t *d_idx, float *d_f, cudaStream_t st)
{
    const int64_t per_cta = (int64_t)PC_COOP_WARPS * (32 / G);
    const int grid = (int)((m + per_cta - 1) / per_cta);
    if (A.kind == PC_Q_NEAREST)
        pc_query_coop_kernel<PC_KIND_NEAREST, G><<<grid, 32 * PC_COOP_WARPS, 0, st>>>(T, A.R, d_q, m, qstride, d_idx, d_f);
    else
        pc_query_coop_kernel<PC_KIND_RADIUS, G><<<grid, 32 * PC_COOP_WARPS, 0, st>>>(T, A.R, d_q, m, qstride, d_idx, d_f);
}

static void pc_launch_coop(const pc_index *ix, const pc_qargs &A, const pc_tree &T, const float *d_q, int64_t m, int qstride,
                           int32_t *d_idx, float *d_f, cudaStream_t st)
{
    int g = ix->coop_group;
    if (g == 0) g = m <= ix->coop_g32_max ? 32 : (m <= ix->coop_g16_max ? 16 : 8);
    if (g == 32) pc_launch_coop_g<32>(A, T, d_q, m, qstride, d_idx, d_f, st);
    else if (g == 16) pc_launch_coop_g<16>(A, T, d_q, m, qstride, d_idx, d_f, st);
    else pc_launch_coop_g<8>(A, T, d_q, m, qstride, d_idx, d_f, st);
}

// Unbounded packet walks are shared by queries within a few packet extents of each other only (pc_query_packet_kernel,
// pc_knn_packet_kernel): 64 queries fill a cube of edge e0 = cell * cbrt(64 / per_cell) at the density of the batch lane L has
// just ordered (cell = 1/256 of the cloud's extent).  Returns ix->packet_split times e0, or 0 (no split).
static float pc_packet_split(const pc_index *ix, const pc_lane &L)
{
    if (!(ix->packet_split > 0.f && L.per_cell > 0.0)) return 0.f;
    float emax = 0.f;
    for (int a = 0; a < 3; a++) { const float e = pc_ordered_to_float(ix->h_bbox[3 + a]) - pc_ordered_to_float(ix->h_bbox[a]); emax = e > emax ? e : emax; }
    const float split = ix->packet_split * (emax / 256.f) * (float)cbrt(64.0 / L.per_cell);
    return split > 0.f ? split : 0.f;
}

// run one device-resident batch on lane L
static int pc_run_batch(pc_index *ix, pc_lane &L, const pc_qargs &A, const float *d_q, int64_t m, int qstride,
                        int32_t *d_idx, float *d_f, bool split_streams = false, bool may_sync = false)
{
    if (m == 0) return PC_OK;
    // Pipelined (ASYNC) batches run their ordering pass on the lane's high-priority stream: its short, memory-bound kernels
    // are scheduled ahead of the queued CTAs of OTHER lanes' search kernels (issue-bound) and overlap with them.  Everything
    // already queued on the lane (input copy, the lane's previous batch, which still reads the sort buffers) comes first.
    const int64_t sort_min = pc_sort_min(ix, A);
    const bool order = pc_want_order(ix, A.flags, m, sort_min);
    L.os = L.stream;
    if (split_streams && order) {
        PC_CUDA(ix, cudaEventRecord(L.ev_deps, L.stream));
        PC_CUDA(ix, cudaStreamWaitEvent(L.order_stream, L.ev_deps, 0));
        L.os = L.order_stream;
    }
    const bool prof = ix->profile && &L == &ix->lane[0];
    if (prof) PC_CUDA(ix, cudaEventRecord(L.t0, L.stream));
    // every batch starts with a zero L.counter (pc_profile_last_deferred_packets); the ordering step clears it when it orders
    if (!order) PC_CUDA(ix, cudaMemsetAsync(L.counter, 0, 2 * sizeof(unsigned long long), L.os));
    pc_order O;
    int rc = pc_order_batch(ix, L, A, sort_min, d_q, nullptr, m, qstride, d_idx, d_f, may_sync, O);
    if (rc != PC_OK) return rc;
    if (L.os != L.stream) {
        PC_CUDA(ix, cudaEventRecord(L.ev_ordered, L.os));
        PC_CUDA(ix, cudaStreamWaitEvent(L.stream, L.ev_ordered, 0));
    }
    if (prof) PC_CUDA(ix, cudaEventRecord(L.t1, L.stream));
    pc_tree T = pc_tree_of(ix);
    // dense batches (>= 3 queries per cell of 1/256 of the cloud's extent): 64-query packets, two queries per lane
    // (profiles/r1_sweep5*: +10 % radius, +18 % nearest at 10 M queries; -3 % at 2 M, hence the threshold)
    const bool two_per_lane = ix->query_kernel == 4 || (ix->query_kernel_auto && L.per_cell >= 3.0);
    const uint32_t *perm = O.perm;
    const float4 *ordered = O.ordered;
    const unsigned long long *m_eff = O.m_eff;
    const bool is_ordered = perm || ordered;
    const int64_t ml = O.m_launch;       // entries the search launch has to cover (the exact share in pc_batch_shard mode)
    // unbounded packet walks put their incoherent packets aside (pc_packet_split)
    pc_radius_dev RN = A.R;
    if ((A.kind == PC_Q_NEAREST || !A.R.bounded) && ix->packet_split > 0.f && L.per_cell > 0.0) {
        RN.packet_split = is_ordered ? pc_packet_split(ix, L) : 0.f;
        RN.defer_count = L.counter;             // zeroed above
        RN.defer_list = L.keys_a;               // the ordering pass is done with its key buffer; one entry per packet at most
    }
    if (ml == 0) {
        // pc_batch_shard: nothing of this batch belongs to this rank
    } else if (is_ordered) {
        // curve-ordered batch: one warp walks the tree once for its 32 or 64 neighbouring queries
        const int per_cta = (two_per_lane ? 2 : 1) * PC_QUERY_THREADS;
        const int grid = (int)((ml + per_cta - 1) / per_cta);
        if (two_per_lane) {
            if (A.kind == PC_Q_NEAREST)
                pc_query_packet_kernel<PC_KIND_NEAREST, 2><<<grid, PC_QUERY_THREADS, 0, L.stream>>>(T, RN, d_q, m, qstride, perm, ordered, m_eff, d_idx, d_f);
            else
                pc_query_packet_kernel<PC_KIND_RADIUS, 2><<<grid, PC_QUERY_THREADS, 0, L.stream>>>(T, RN, d_q, m, qstride, perm, ordered, m_eff, d_idx, d_f);
        } else if (A.kind == PC_Q_NEAREST)
            pc_query_packet_kernel<PC_KIND_NEAREST, 1><<<grid, PC_QUERY_THREADS, 0, L.stream>>>(T, RN, d_q, m, qstride, perm, ordered, m_eff, d_idx, d_f);
        else
            pc_query_packet_kernel<PC_KIND_RADIUS, 1><<<grid, PC_QUERY_THREADS, 0, L.stream>>>(T, RN, d_q, m, qstride, perm, ordered, m_eff, d_idx, d_f);
    } else if (m <= ((A.kind == PC_Q_NEAREST || !A.R.bounded) ? ix->coop_max_unbounded : ix->coop_max)) {
        // small unordered batch: one warp per query (a thread-per-query search is a chain of dependent loads)
        pc_launch_coop(ix, A, T, d_q, m, qstride, d_idx, d_f, L.stream);
    } else {
        const int grid = (int)((m + PC_QUERY_THREADS - 1) / PC_QUERY_THREADS);
        if (A.kind == PC_Q_NEAREST)
            pc_query_simple_kernel<PC_KIND_NEAREST><<<grid, PC_QUERY_THREADS, 0, L.stream>>>(T, A.R, d_q, m, qstride, d_idx, d_f);
        else
            pc_query_simple_kernel<PC_KIND_RADIUS><<<grid, PC_QUERY_THREADS, 0, L.stream>>>(T, A.R, d_q, m, qstride, d_idx, d_f);
    }
    if (ml > 0) ix->launches++;
    if (is_ordered && ml > 0 && RN.packet_split > 0.f) {
        // the packets the walk above put aside as incoherent (normally none or a handful: the kernel then costs its launch)
        const int dgrid = ix->sm_count * PC_DEFER_CTAS_PER_SM;
        const int per_packet = (two_per_lane ? 2 : 1) * 32;
        if (A.kind == PC_Q_NEAREST) pc_query_deferred_kernel<PC_KIND_NEAREST><<<dgrid, PC_QUERY_THREADS, 0, L.stream>>>(T, RN, d_q, m, qstride, per_packet, perm, ordered, m_eff, d_idx, d_f);
        else pc_query_deferred_kernel<PC_KIND_RADIUS><<<dgrid, PC_QUERY_THREADS, 0, L.stream>>>(T, RN, d_q, m, qstride, per_packet, perm, ordered, m_eff, d_idx, d_f);
        ix->launches++;
    }
    PC_CHECK_LAUNCH(ix);
    if (prof) { PC_CUDA(ix, cudaEventRecord(L.t2, L.stream)); ix->profiled = true; }
    return PC_OK;
}

// One PC_HOST chunk on lane L: rows [off, off + c) of `width` outputs each.  The lane's output buffers grow to hold the chunk
// (at least `rows` rows), run(L, off, c, d_idx, d_f) stages the chunk's inputs on the lane and runs them into d_idx / d_f, and
// the rows go home on the lane's stream.
template <class RUN>
static int pc_host_chunk(pc_index *ix, pc_lane &L, int64_t off, int64_t c, int64_t rows, int64_t width, int32_t *out_idx, float *out_f,
                         RUN &run)
{
    int rc;
    if (out_idx && (rc = pc_grow(ix, &L.d_i32, &L.i32_cap, c * width, rows * width)) != PC_OK) return rc;
    if (out_f && (rc = pc_grow(ix, &L.d_f32, &L.f32_cap, c * width, rows * width)) != PC_OK) return rc;
    if ((rc = run(L, off, c, out_idx ? L.d_i32 : nullptr, out_f ? L.d_f32 : nullptr)) != PC_OK) return rc;
    if (out_idx) PC_CUDA(ix, cudaMemcpyAsync(out_idx + off * width, L.d_i32, (size_t)c * width * sizeof(int32_t), cudaMemcpyDeviceToHost, L.stream));
    if (out_f) PC_CUDA(ix, cudaMemcpyAsync(out_f + off * width, L.d_f32, (size_t)c * width * sizeof(float), cudaMemcpyDeviceToHost, L.stream));
    return PC_OK;
}

// Blocking PC_HOST batches of the row-per-query calls: chunks of `chunk` rows over the pipeline lanes (pc_host_chunk), after
// the last index build on the handle's stream.  A multi-chunk call sizes the lane buffers for full chunks at once; a small
// call allocates only what it needs.
template <class RUN>
static int pc_host_chunks(pc_index *ix, int64_t m, int64_t chunk, int64_t width, int32_t *out_idx, float *out_f, RUN run)
{
    for (int l = 1; l < PC_PIPE_LANES; l++) PC_CUDA(ix, cudaStreamWaitEvent(ix->lane[l].stream, ix->ev_ready, 0));
    const int64_t rows = m > chunk ? chunk : 0;
    int li = 0;
    for (int64_t off = 0; off < m; off += chunk, li = (li + 1) % PC_PIPE_LANES) {
        int rc = pc_host_chunk(ix, ix->lane[li], off, m - off < chunk ? m - off : chunk, rows, width, out_idx, out_f, run);
        if (rc != PC_OK) return rc;
    }
    for (int l = 0; l < PC_PIPE_LANES; l++) PC_CUDA(ix, cudaStreamSynchronize(ix->lane[l].stream));
    return PC_OK;
}

extern "C" int pc_batch_shard(pc_index *ix, int rank, int n_ranks)
{
    if (!ix || n_ranks < 1 || rank < 0 || rank >= n_ranks) return pc_fail(ix, PC_EINVAL, "pc_batch_shard: bad argument");
    if (n_ranks > 1 && ix->sort_bits == 0)
        return pc_fail(ix, PC_EINVAL, "pc_batch_shard: the share is selected by the ordering pass, which PC_SORT_BITS=0 disabled");
    ix->shard_rank = rank;
    ix->shard_n = n_ranks;
    return PC_OK;
}

extern "C" int pc_index_set_radius_arith(pc_index *ix, int mode)
{
    if (!ix || (mode != PC_ARITH_FP64 && mode != PC_ARITH_PCL_FLOAT)) return pc_fail(ix, PC_EINVAL, "pc_index_set_radius_arith: bad argument");
    ix->radius_arith = mode;
    return PC_OK;
}

extern "C" int pc_profile_enable(pc_index *ix, int on)
{
    if (!ix) return PC_EINVAL;
    ix->profile = on != 0;
    ix->profiled = false;
    return PC_OK;
}

// detail of the ordering pass of the last profiled, ORDERED PC_DEVICE batch: out[0] = clearing the sort scratch, out[1] = key
// kernel (curve keys, early-outs, compaction, digit histograms), out[2] = the radix sort passes
extern "C" int pc_profile_last_order_detail(pc_index *ix, float out[3])
{
    if (!ix || !out) return PC_EINVAL;
    if (!ix->profiled) return pc_fail(ix, PC_EINVAL, "pc_profile_last_order_detail: no profiled PC_DEVICE batch yet");
    PC_CUDA(ix, cudaSetDevice(ix->device));
    pc_lane &L = ix->lane[0];
    PC_CUDA(ix, cudaEventSynchronize(L.t2));
    if (cudaEventElapsedTime(&out[0], L.t0, L.ta) != cudaSuccess || cudaEventElapsedTime(&out[1], L.ta, L.tb) != cudaSuccess ||
        cudaEventElapsedTime(&out[2], L.tb, L.t1) != cudaSuccess) {
        cudaGetLastError();
        return pc_fail(ix, PC_EINVAL, "pc_profile_last_order_detail: the last batch was not ordered");
    }
    return PC_OK;
}

extern "C" int pc_profile_last_deferred_packets(pc_index *ix, int64_t *packets)
{
    if (!ix || !packets) return PC_EINVAL;
    PC_CUDA(ix, cudaSetDevice(ix->device));
    pc_lane &L = ix->lane[0];
    unsigned long long h = 0;
    // counter[0] of the lane: zeroed at the start of every batch, bumped by the unbounded pc_query_packet_kernel walks only
    PC_CUDA(ix, cudaMemcpyAsync(&h, L.counter, sizeof h, cudaMemcpyDeviceToHost, L.stream));
    PC_CUDA(ix, cudaStreamSynchronize(L.stream));
    *packets = (int64_t)h;
    return PC_OK;
}

extern "C" int pc_profile_last_batch(pc_index *ix, float *order_ms, float *search_ms)
{
    if (!ix) return PC_EINVAL;
    if (!ix->profiled) return pc_fail(ix, PC_EINVAL, "pc_profile_last_batch: no profiled PC_DEVICE batch yet");
    PC_CUDA(ix, cudaSetDevice(ix->device));
    pc_lane &L = ix->lane[0];
    PC_CUDA(ix, cudaEventSynchronize(L.t2));
    float a = 0.f, b = 0.f;
    PC_CUDA(ix, cudaEventElapsedTime(&a, L.t0, L.t1));
    PC_CUDA(ix, cudaEventElapsedTime(&b, L.t1, L.t2));
    if (order_ms) *order_ms = a;
    if (search_ms) *search_ms = b;
    return PC_OK;
}

// Blocking PC_HOST call with a handful of queries -- what the unmodified planner loop issues (one radiusSearch per RRT*
// iteration, corridor_finder.cpp:404).  Two staged copies plus three stream syncs cost ~65 us per call; here the
// kernel reads the queries from, and writes the results to, pinned host memory mapped into the device's address space
// (a few PCIe transactions), so a call is one launch and one sync on the handle's stream, and the kernel puts a whole warp on
// every query (pc_query_coop_kernel).
static int pc_tiny_host_batch(pc_index *ix, const pc_qargs &A, const float *q, int64_t m, int qs, int32_t *out_idx, float *out_f)
{
    memcpy(ix->tiny_q, q, (size_t)m * qs * sizeof(float));
    pc_tree T = pc_tree_of(ix);
    int32_t *d_i = out_idx ? ix->tiny_i_dev : nullptr;
    float *d_f = out_f ? ix->tiny_f_dev : nullptr;
    // one warp per query: the search of a single query is a chain of dependent loads, the warp shortens it
    pc_launch_coop(ix, A, T, ix->tiny_q_dev, m, qs, d_i, d_f, ix->stream);
    ix->launches++;
    PC_CHECK_LAUNCH(ix);
    PC_CUDA(ix, cudaStreamSynchronize(ix->stream));
    if (out_idx) memcpy(out_idx, ix->tiny_i, (size_t)m * sizeof(int32_t));
    if (out_f) memcpy(out_f, ix->tiny_f, (size_t)m * sizeof(float));
    return PC_OK;
}

// PC_HOST: chunked pipeline over the lanes; PC_DEVICE: one batch on the handle's stream
static int pc_query_dispatch(pc_index *ix, const pc_qargs &A, const float *q, int64_t m, int64_t q_stride, int space,
                             int32_t *out_idx, float *out_f)
{
    PC_CUDA(ix, cudaSetDevice(ix->device));
    if (m == 0) return PC_OK;
    const int qs = (int)q_stride;
    if (space == PC_DEVICE) return pc_run_batch(ix, ix->lane[0], A, q, m, qs, out_idx, out_f, false, true);
    if (space == PC_HOST && m <= ix->tiny_batch && !pc_want_order(ix, A.flags, m, pc_sort_min(ix, A))) return pc_tiny_host_batch(ix, A, q, m, qs, out_idx, out_f);

    // PC_HOST: the queries staged per chunk, and on a pc_batch_shard handle the caller's current outputs too (the entries of
    // other ranks' queries must come back untouched); PC_HOST_ASYNC: the whole batch as one such chunk (below)
    auto run = [&](pc_lane &L, int64_t off, int64_t c, int32_t *d_idx, float *d_f) {
        // (a chunk of a multi-chunk call: room for a full chunk of 4-float rows at once, as pc_host_chunks gives the outputs)
        int rc = pc_grow(ix, &L.d_q, &L.q_cap, c * qs, c < m ? ix->host_chunk * 4 : 0);
        if (rc != PC_OK) return rc;
        PC_CUDA(ix, cudaMemcpyAsync(L.d_q, q + off * qs, (size_t)c * qs * sizeof(float), cudaMemcpyHostToDevice, L.stream));
        if (ix->shard_n > 1) {
            if (d_idx) PC_CUDA(ix, cudaMemcpyAsync(d_idx, out_idx + off, (size_t)c * sizeof(int32_t), cudaMemcpyHostToDevice, L.stream));
            if (d_f) PC_CUDA(ix, cudaMemcpyAsync(d_f, out_f + off, (size_t)c * sizeof(float), cudaMemcpyHostToDevice, L.stream));
        }
        return pc_run_batch(ix, L, A, L.d_q, c, qs, d_idx, d_f, space == PC_HOST_ASYNC);
    };
    if (space == PC_HOST) return pc_host_chunks(ix, m, ix->host_chunk, 1, out_idx, out_f, run);

    // order the side lanes after the last (possibly still running) index build / broadcast on the handle's stream
    for (int l = 1; l < PC_PIPE_LANES; l++) PC_CUDA(ix, cudaStreamWaitEvent(ix->lane[l].stream, ix->ev_ready, 0));
    pc_lane &L = ix->lane[ix->next_lane];
    ix->next_lane = (ix->next_lane + 1) % PC_PIPE_LANES;
    int rc;
    if (space == PC_DEVICE_ASYNC) {
        // device-resident batch on the next lane: consecutive calls overlap one batch's ordering pass (memory-bound) with the
        // previous batch's search (issue-bound).  The lane starts after whatever the handle's stream holds now (the
        // caller's producers of q); results are valid after pc_index_sync.
        if (&L != &ix->lane[0]) {
            PC_CUDA(ix, cudaEventRecord(ix->ev_in, ix->stream));
            PC_CUDA(ix, cudaStreamWaitEvent(L.stream, ix->ev_in, 0));
        }
        rc = pc_run_batch(ix, L, A, q, m, qs, out_idx, out_f, true);
    } else {
        // PC_HOST_ASYNC: the whole batch on the next lane, no wait: consecutive calls overlap their H2D / kernels / D2H
        rc = pc_host_chunk(ix, L, 0, m, 0, 1, out_idx, out_f, run);
    }
    if (rc != PC_OK) return rc;
    PC_CUDA(ix, cudaEventRecord(L.done, L.stream));      // a later rebuild must wait for this batch
    return PC_OK;
}

static int pc_check_query_args(pc_index *ix, const char *fn, const float *q, int64_t m, int64_t q_stride, int space)
{
    if (!ix) return PC_EINVAL;
    if (m < 0 || (m > 0 && !q) || (q_stride != 3 && q_stride != 4) || (space != PC_HOST && space != PC_DEVICE && space != PC_HOST_ASYNC && space != PC_DEVICE_ASYNC))
        return pc_fail(ix, PC_EINVAL, "%s: bad argument (m=%lld stride=%lld space=%d)", fn, (long long)m, (long long)q_stride, space);
    if (m > ((int64_t)1 << 32) - 1) return pc_fail(ix, PC_EINVAL, "%s: at most 2^32-1 queries per call", fn);
    return PC_OK;
}

extern "C" int pc_nearest_batch(pc_index *ix, const float *q_xyz, int64_t m, int64_t q_stride, int space, int flags,
                                int32_t *out_idx, float *out_d2)
{
    int rc = pc_check_query_args(ix, "pc_nearest_batch", q_xyz, m, q_stride, space);
    if (rc != PC_OK) return rc;
    return pc_query_dispatch(ix, pc_nearest_qargs(flags), q_xyz, m, q_stride, space, out_idx, out_d2);
}

static int pc_make_radius_dev(pc_index *ix, const pc_radius_params *p, int flags, pc_radius_dev *R)
{
    if (!p || !(p->max_radius == p->max_radius) || !(p->search_margin == p->search_margin))
        return pc_fail(ix, PC_EINVAL, "pc_radius_params: null or NaN");
    R->search_margin = p->search_margin; R->max_radius = p->max_radius; R->sample_range = p->sample_range;
    R->sx = p->start[0]; R->sy = p->start[1]; R->sz = p->start[2];
    R->bounded = (flags & PC_RADIUS_FULL_NN) ? 0 : 1;
    R->pcl_float = ix->radius_arith == PC_ARITH_PCL_FLOAT ? 1 : 0;
    {
        const double T = p->sample_range + p->max_radius, t2 = T * T;
        R->range_lo2 = T > 0.0 ? t2 * (1.0 - 1e-12) : -1.0;       // T <= 0: always the exact expression
        R->range_hi2 = T > 0.0 ? t2 * (1.0 + 1e-12) : INFINITY;
    }
    R->bound_thr = FLT_MAX;
    if (R->bounded) {
        // radius = min(sqrt(d2) - margin, max_radius): every d > max_radius + margin gives max_radius, so the search
        // may stop there.  1e-6 relative head-room keeps the clamp decision exact in fp64.
        double bound = (p->max_radius + p->search_margin) * (1.0 + 1e-6);
        if (bound < 0.0) bound = 0.0;
        double b2 = bound * bound * (1.0 + 1e-6);
        float f = (float)b2;
        f = nextafterf(f, INFINITY) * PC_THR_SLACK;
        R->bound_thr = f < FLT_MAX ? f : FLT_MAX;
    }
    return PC_OK;
}

extern "C" int pc_radius_batch(pc_index *ix, const float *q_xyz, int64_t m, int64_t q_stride, int space, int flags,
                               const pc_radius_params *params, float *out_radius, int32_t *out_idx)
{
    int rc = pc_check_query_args(ix, "pc_radius_batch", q_xyz, m, q_stride, space);
    if (rc != PC_OK) return rc;
    pc_qargs A;
    memset(&A, 0, sizeof A);
    A.kind = PC_Q_RADIUS; A.flags = flags;
    if ((rc = pc_make_radius_dev(ix, params, flags, &A.R)) != PC_OK) return rc;
    return pc_query_dispatch(ix, A, q_xyz, m, q_stride, space, out_idx, out_radius);
}

#include "range_host.inl"
#include "range_sorted_host.inl"
#include "knn_host.inl"
#include "knn_large_host.inl"
#include "field_host.inl"
#include "segment_host.inl"
#include "sweep_host.inl"
#include "clearance_host.inl"
#include "traj_sweep_host.inl"
#include "traj_nearest_host.inl"
#include "sampler_host.inl"
#include "comm_host.inl"
#include "kd_compat.inl"

#ifdef PC_STATS
extern "C" int pc_stats_read(unsigned long long out[65], int reset)
{
    if (cudaMemcpyFromSymbol(out, pc_stats_hist, 65 * sizeof(unsigned long long)) != cudaSuccess) return PC_ECUDA;
    if (reset) { unsigned long long z[65] = { 0 }; cudaMemcpyToSymbol(pc_stats_hist, z, sizeof z); }
    return PC_OK;
}
#endif
