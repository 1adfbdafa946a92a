// mpp_astar.cu -- batched A* connectors, waypoint-chain fitness (PSO/GA) and path statistics.
// Reference semantics: astar.py:33-101, MPA.py:106-151, helper.py:58-113, MPA.py:176-229,
// pso.py:56-94, ga_solver.py:58-93.
#include <cmath>
#include <vector>

#include "mpp_astar.cuh"
#include "mpp_stats.cuh"

#define MPP_AS_THREADS (MPP_GL == 32 ? 256 : 128)
#define MPP_AS_WARPS (MPP_AS_THREADS / 32)
#define MPP_AS_GROUPS (MPP_AS_THREADS / MPP_GL)     // searches (lane groups) per CTA

// ---------------------------------------------------------------------------------------------
// K1b: safety-class table (helper.py:67-80 as a per-cell function of the map)
//   class[cell] = min squared distance to an obstacle within the (2*radius+1)^2 stencil, radius = floor(msd); 0 = none.
//   lut[d2]     = (msd - sqrt(d2))**2 if sqrt(d2) < msd else 0   -- evaluated on the host with libm pow.
// Only obstacles nearer than msd contribute (helper.py:76), and those lie inside the stencil.
// Out-of-bounds is NOT an obstacle here (obstacle_nodes = argwhere(grid == 1), helper.py:125).
// ---------------------------------------------------------------------------------------------
__global__ void mpp_safety_kernel(const uint32_t *__restrict__ occ, int occ_words, int pitch, int R, int C, int radius,
                                  uint16_t *__restrict__ cls) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * C) return;
    occ += (size_t)blockIdx.y * occ_words;                     // blockIdx.y = map of a batch
    cls += (size_t)blockIdx.y * R * C;
    const int r = i / C, c = i % C;
    int best = 1 << 30;
    for (int dr = -radius; dr <= radius; ++dr) {
        const int rr = r + dr;
        if (rr < 0 || rr >= R) continue;
        for (int dc = -radius; dc <= radius; ++dc) {
            const int c2 = c + dc;
            if (c2 < 0 || c2 >= C) continue;
            const int pb = c2 + 1;
            if ((occ[(rr + 1) * pitch + (pb >> 5)] >> (pb & 31)) & 1u) {
                const int d2 = dr * dr + dc * dc;
                best = d2 < best ? d2 : best;
            }
        }
    }
    cls[i] = (best == (1 << 30)) ? 0 : (uint16_t)best;          // best <= 2*radius^2 < 65536 (radius <= 180)
}

extern "C" int mpp_map_batch_safety_table(mpp_map_batch *maps, double msd, void *stream) {
    MPP_REQUIRE(maps, "mpp_map_batch_safety_table: null batch");
    MPP_REQUIRE(msd >= 0.0 && msd <= 180.0, "mpp_map_batch_safety_table: min_safe_distance %g unsupported (0 <= msd <= 180)", msd);
    if (maps->safety_msd == msd && maps->safety_d2_dev) return MPP_OK;
    MPP_CUDA(cudaSetDevice(maps->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int n = maps->rows * maps->cols;
    const int radius = (int)msd;                               // an obstacle nearer than msd has |dr|, |dc| <= floor(msd)
    const int need = 2 * radius * radius + 2;
    if (!maps->safety_d2_dev) MPP_CUDA(cudaMalloc(&maps->safety_d2_dev, (size_t)n * maps->n_maps * sizeof(uint16_t)));
    if (maps->safety_lut_n < need) {
        MPP_CUDA(cudaStreamSynchronize(s));                     // a kernel of an earlier call may still read the old table
        if (maps->safety_lut_dev) MPP_CUDA(cudaFree(maps->safety_lut_dev));
        maps->safety_lut_dev = nullptr;
        MPP_CUDA(cudaMalloc(&maps->safety_lut_dev, (size_t)need * sizeof(double)));
        maps->safety_lut_n = need;
    }
    std::vector<double> h((size_t)need, 0.0);
    for (int k = 1; k < need; ++k) {
        const double d = std::sqrt((double)k);
        h[k] = (d < msd) ? std::pow(msd - d, 2.0) : 0.0;        // helper.py:77-78 (float ** 2 -> libm pow)
    }
    MPP_CUDA(cudaMemcpyAsync(maps->safety_lut_dev, h.data(), (size_t)need * sizeof(double), cudaMemcpyHostToDevice, s));
    MPP_CUDA(cudaStreamSynchronize(s));
    mpp_safety_kernel<<<dim3((n + 255) / 256, maps->n_maps), 256, 0, s>>>(maps->occ_dev, maps->occ_words, maps->pitch_words,
                                                                          maps->rows, maps->cols, radius, maps->safety_d2_dev);
    MPP_CUDA(cudaGetLastError());
    maps->safety_msd = msd;
    return MPP_OK;
}

int mpp_stats_ctx(mpp_map_batch *maps, const mpp_policy *pol, void *stream, StatsCtx *X) {
    X->occ = maps->occ_dev; X->pitch = maps->pitch_words; X->R = maps->rows; X->C = maps->cols;
    X->pol = *pol;
    X->cls = nullptr; X->lut = nullptr;
    if (pol->mode == 0 && maps->n_obstacles > 0) {             // an obstacle-free map's classes are all 0 (penalty 0.0)
        const int rc = mpp_map_batch_safety_table(maps, pol->min_safe_distance, stream);
        if (rc) return rc;
        X->cls = maps->safety_d2_dev; X->lut = maps->safety_lut_dev;
    }
    return MPP_OK;
}

__global__ void __launch_bounds__(MPP_AS_THREADS)
mpp_path_stats_kernel(StatsCtx X, int occ_words, int n_maps, const int32_t *__restrict__ map,
                      const int32_t *__restrict__ cells, int max_cells, const int32_t *__restrict__ n_cells, int n_paths,
                      double *stats) {
    const LaneGroup L = lane_group();
    const int w = (blockIdx.x * MPP_AS_THREADS + threadIdx.x) / MPP_GL;
    if (w >= n_paths) return;
    const int m = map[w];
    int n = n_cells[w];
    if (n > max_cells) n = max_cells;
    if ((unsigned)m < (unsigned)n_maps) {
        X.occ += (size_t)m * occ_words;
        if (X.cls) X.cls += (size_t)m * X.R * X.C;
    } else {
        n = 0;                                                  // outside the batch: the empty path's statistics
    }
    path_stats_warp(L, X, cells + (size_t)w * max_cells, n, stats + (size_t)w * 5);
}

extern "C" int mpp_path_stats(mpp_map_batch *maps, const int32_t *map_dev, const int32_t *cells_dev, int max_cells,
                              const int32_t *n_cells_dev, int n_paths, const mpp_policy *policy, double *stats_dev,
                              void *stream) {
    MPP_REQUIRE(maps && map_dev && cells_dev && n_cells_dev && policy && stats_dev, "mpp_path_stats: null argument");
    MPP_REQUIRE(n_paths > 0 && max_cells > 0, "mpp_path_stats: bad sizes");
    MPP_CUDA(cudaSetDevice(maps->device));
    StatsCtx X;
    int rc = mpp_stats_ctx(maps, policy, stream, &X);
    if (rc) return rc;
    const int blocks = (n_paths + MPP_AS_GROUPS - 1) / MPP_AS_GROUPS;
    mpp_path_stats_kernel<<<blocks, MPP_AS_THREADS, 0, (cudaStream_t)stream>>>(X, maps->occ_words, maps->n_maps, map_dev,
                                                                             cells_dev, max_cells, n_cells_dev, n_paths,
                                                                             stats_dev);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

// ---------------------------------------------------------------------------------------------
// scratch layout: [0,256) work counter + error flag; then n_slots search slots
// ---------------------------------------------------------------------------------------------
extern "C" size_t mpp_astar_slot_bytes(int rows, int cols, int heap_cap) {
    if (rows <= 0 || cols <= 0 || heap_cap <= 0) return 0;
    return astar_slot_bytes(rows * cols, heap_cap);
}

// search slots (lane groups) that are resident at once: three CTAs of MPP_AS_GROUPS groups per SM
extern "C" int mpp_map_batch_max_slots(const mpp_map_batch *maps) { return maps ? maps->sm_count * 3 * MPP_AS_GROUPS : 0; }

static int check_search(const mpp_map_batch *maps, size_t scratch_bytes, int n_slots, int heap_cap) {
    // the searches pack a node as (row << 16 | col) in a signed int (same (r, c) order as the reference's tuples)
    MPP_REQUIRE(maps->rows < 32768 && maps->cols < 65536,
                "A*: map %dx%d exceeds the packed-node limit (rows < 32768, cols < 65536)", maps->rows, maps->cols);
    MPP_REQUIRE(n_slots > 0 && heap_cap >= 64, "A*: n_slots=%d heap_cap=%d", n_slots, heap_cap);
    const size_t need = 256 + (size_t)n_slots * astar_slot_bytes(maps->rows * maps->cols, heap_cap);
    MPP_REQUIRE(scratch_bytes >= need, "A*: scratch too small (%zu < %zu)", scratch_bytes, need);
    return MPP_OK;
}

int mpp_occ_staging(const void *kernel, MppStaging &st, int device, size_t occ_bytes, bool *stage) {
    *stage = occ_bytes <= MPP_OCC_STAGE_MAX;
    if (!*stage) return MPP_OK;
    if (st.static_bytes < 0) {
        cudaFuncAttributes fa;
        MPP_CUDA(cudaFuncGetAttributes(&fa, kernel));
        st.static_bytes = (int)fa.sharedSizeBytes;
    }
    const int dv = device & 63;
    if ((size_t)st.static_bytes + occ_bytes > 48 * 1024 && (int)occ_bytes > st.raised[dv]) {
        MPP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)occ_bytes));
        st.raised[dv] = (int)occ_bytes;
    }
    return MPP_OK;
}

// The search and fitness kernels stage the occupancy of a one-map batch in shared memory when it fits (their <true>
// instantiations); a larger map, or a batch of several maps, is read through L2.
static int stage_one_map(const void *staged_kernel, MppStaging &st, const mpp_map_batch *maps, bool *stage) {
    *stage = false;
    if (maps->n_maps != 1) return MPP_OK;
    return mpp_occ_staging(staged_kernel, st, maps->device, (size_t)maps->occ_words * 4, stage);
}

struct SearchArgs {
    AStarGrid G;            // G.occ: [n_maps][occ_words] occupancy
    int occ_words;
    int variant;
    const int32_t *map, *src, *dst;   // query i: map[i], src[i] -> dst[i]
    const uint32_t *avoid;  // n x words or null
    int n, n_maps, words;
    int32_t *cells;
    int max_cells;
    int32_t *n_cells;
    double *g;
    char *scratch;
    int n_slots, heap_cap;
    unsigned long long *counters;
    const int32_t *order;   // optional processing order of the queries (null: index order)
    StatsCtx X;             // statistics of each found path (X.cls: [n_maps][R*C] safety classes or null)
    double *stats;          // n x 5, or null: no statistics
};

// Query i on map A.map[i], read through that map's slice of global memory (L2) or, OCC_SMEM (a one-map batch), from
// the copy staged in shared memory; with A.stats, the statistics of its path computed by the same lane group right after
// the search.
template <bool OCC_SMEM>
__global__ void __launch_bounds__(MPP_AS_THREADS, 3) mpp_astar_batch_kernel(SearchArgs A) {
    extern __shared__ __align__(16) uint32_t s_occ[];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ __align__(16) uint8_t s_cnt[MPP_AS_GROUPS][MPP_PQ_NB];
    if (OCC_SMEM) mpp_stage_bulk(s_occ, A.G.occ, (uint32_t)A.occ_words * 4u, &s_bar);
    const LaneGroup L = lane_group();
    const int lane = L.gl;
    const int slot = (blockIdx.x * MPP_AS_THREADS + threadIdx.x) / MPP_GL;
    if (slot >= A.n_slots) return;
    const int rc = A.G.R * A.G.C;
    AStarSlot S = astar_slot_at(A.scratch + 256 + (size_t)slot * astar_slot_bytes(rc, A.heap_cap), rc, A.heap_cap,
                                s_cnt[threadIdx.x / MPP_GL]);
    unsigned int *next = (unsigned int *)A.scratch;
    for (;;) {
        int i = 0;
        if (lane == 0) i = (int)atomicAdd(next, 1u);
        i = grp_shfl(L, i, 0);
        if (i >= A.n) break;
        if (A.order) i = A.order[i];                                   // longest queries first (see mpp_astar_batch_maps)
        const int m = A.map[i], src = A.src[i], dst = A.dst[i];
        int32_t *path = A.cells + (size_t)i * A.max_cells;
        int len = 0;
        double g = __longlong_as_double(MPP_INF_BITS);
        AStarGrid Gm = A.G;
        Gm.occ = OCC_SMEM ? s_occ : A.G.occ + (size_t)m * A.occ_words;   // (staged: the batch's one map)
        if ((unsigned)m < (unsigned)A.n_maps && (unsigned)src < (unsigned)rc && (unsigned)dst < (unsigned)rc)
            len = astar_search(L, Gm, S, A.variant, src, dst, A.avoid ? A.avoid + (size_t)i * A.words : nullptr, path,
                               A.max_cells, &g, A.counters);
        if (lane == 0) { A.n_cells[i] = len; if (A.g) A.g[i] = g; }
        if (A.stats) {                                                 // helper.py:98-113 on the path just found
            StatsCtx X = A.X;
            X.occ = Gm.occ;
            if (X.cls) X.cls += (size_t)m * rc;
            path_stats_warp(L, X, path, (len > 0 && len <= A.max_cells) ? len : 0, A.stats + (size_t)i * 5);
        }
    }
}

// Queries over a batch of same-shape maps (query i on map map_dev[i]), the statistics of each path fused in.
extern "C" int mpp_astar_batch_maps(mpp_map_batch *maps, int variant, const int32_t *map_dev, const int32_t *src_dev,
                                    const int32_t *dst_dev, const uint32_t *avoid_bits_dev, int n, int allow_diagonal,
                                    int restrict_corner, const mpp_policy *stats_policy, int32_t *cells_dev, int max_cells,
                                    int32_t *n_cells_dev, double *g_dev, double *stats_dev, void *scratch_dev,
                                    size_t scratch_bytes, int n_slots, int heap_cap, unsigned long long *counters_dev,
                                    const int32_t *order_dev, void *stream) {
    MPP_REQUIRE(maps && map_dev && src_dev && dst_dev && cells_dev && n_cells_dev && scratch_dev,
                "mpp_astar_batch_maps: null argument");
    MPP_REQUIRE(!stats_policy || stats_dev, "mpp_astar_batch_maps: stats_policy without stats_dev");
    MPP_REQUIRE(variant >= 0 && variant <= 2, "mpp_astar_batch_maps: variant must be 0 (astar.py), 1 (MPA.py) or 2 (dijkstra.py)");
    MPP_REQUIRE(n > 0 && max_cells > 0, "mpp_astar_batch_maps: bad sizes");
    int rc = check_search(maps, scratch_bytes, n_slots, heap_cap);
    if (rc) return rc;
    MPP_CUDA(cudaSetDevice(maps->device));
    cudaStream_t s = (cudaStream_t)stream;
    SearchArgs A;
    memset(&A, 0, sizeof(A));
    if (stats_policy) {
        rc = mpp_stats_ctx(maps, stats_policy, stream, &A.X);
        if (rc) return rc;
        A.stats = stats_dev;
    }
    MPP_CUDA(cudaMemsetAsync(scratch_dev, 0, 256, s));
    A.G.occ = maps->occ_dev; A.G.pitch = maps->pitch_words; A.G.R = maps->rows; A.G.C = maps->cols;
    A.G.allow_diag = allow_diagonal; A.G.restrict_corner = restrict_corner;
    A.occ_words = maps->occ_words; A.variant = variant; A.map = map_dev; A.src = src_dev; A.dst = dst_dev;
    A.avoid = avoid_bits_dev; A.n = n; A.n_maps = maps->n_maps; A.words = (maps->rows * maps->cols + 31) / 32;
    A.cells = cells_dev; A.max_cells = max_cells; A.n_cells = n_cells_dev; A.g = g_dev; A.scratch = (char *)scratch_dev;
    A.n_slots = n_slots; A.heap_cap = heap_cap; A.counters = counters_dev; A.order = order_dev;
    const int blocks = (n_slots + MPP_AS_GROUPS - 1) / MPP_AS_GROUPS;
    static MppStaging staging = {-1, {0}};
    bool stage;
    rc = stage_one_map((const void *)mpp_astar_batch_kernel<true>, staging, maps, &stage);
    if (rc) return rc;
    if (stage) mpp_astar_batch_kernel<true><<<blocks, MPP_AS_THREADS, (size_t)maps->occ_words * 4, s>>>(A);
    else mpp_astar_batch_kernel<false><<<blocks, MPP_AS_THREADS, 0, s>>>(A);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

// ---------------------------------------------------------------------------------------------
// K6 + K7: waypoint chain -> path -> fitness (pso.py:56-94 / ga_solver.py:58-93 + helper.py:98-113)
// One warp per individual: W+1 sequential connector searches with the growing avoid set
// (nodes_in_path_so_far - {current_start, waypoint}), then the statistics of the joined path.
// n_cells: 0 = invalid individual ([]), -1 = heap overflow, > max_cells = path truncated.
// ---------------------------------------------------------------------------------------------
struct ChainArgs {
    AStarGrid G;             // G.occ: [n_maps][occ_words] occupancy
    int occ_words;
    StatsCtx X;              // X.cls: [n_maps][R*C] safety classes or null
    const int32_t *map;      // individual i runs on map map[i] ...
    int n_maps;
    const MppMapMeta *meta;  // ... from meta[map[i]].start to meta[map[i]].target
    const int32_t *wps;      // N x W cells
    int N, W, words;
    int32_t *cells;
    int max_cells;
    int32_t *n_cells;
    double *stats;
    uint32_t *visited;       // n_slots x words
    char *scratch;
    int n_slots, heap_cap;
    unsigned long long *counters;
    const int32_t *order;    // optional processing order of the individuals (null: index order)
};

// Individual i on map A.map[i] from that map's start to its target, the occupancy read as mpp_astar_batch_kernel reads
// it, its statistics from that map's safety classes.
template <bool OCC_SMEM>
__global__ void __launch_bounds__(MPP_AS_THREADS, 3) mpp_waypoint_fitness_kernel(ChainArgs A) {
    extern __shared__ __align__(16) uint32_t s_occ[];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ __align__(16) uint8_t s_cnt[MPP_AS_GROUPS][MPP_PQ_NB];
    if (OCC_SMEM) mpp_stage_bulk(s_occ, A.G.occ, (uint32_t)A.occ_words * 4u, &s_bar);
    const LaneGroup L = lane_group();
    const int lane = L.gl;
    const int slot = (blockIdx.x * MPP_AS_THREADS + threadIdx.x) / MPP_GL;
    if (slot >= A.n_slots) return;
    const int rc = A.G.R * A.G.C;
    AStarSlot S = astar_slot_at(A.scratch + 256 + (size_t)slot * astar_slot_bytes(rc, A.heap_cap), rc, A.heap_cap,
                                s_cnt[threadIdx.x / MPP_GL]);
    unsigned int *next = (unsigned int *)A.scratch;
    uint32_t *vis = A.visited + (size_t)slot * A.words;               // a slot runs one chain at a time
    for (;;) {
        int i = 0;
        if (lane == 0) i = (int)atomicAdd(next, 1u);
        i = grp_shfl(L, i, 0);
        if (i >= A.N) break;
        if (A.order) i = A.order[i];                                   // longest chains first (see mpp_waypoint_fitness_maps)
        const int m = A.map[i];
        int start = -1, target = -1;
        if ((unsigned)m < (unsigned)A.n_maps) { start = A.meta[m].start; target = A.meta[m].target; }
        int32_t *path = A.cells + (size_t)i * A.max_cells;
        if (start < 0 || target < 0) {                                 // outside the batch: not searched
            if (lane == 0) A.n_cells[i] = 0;
            path_stats_warp(L, A.X, path, 0, A.stats + (size_t)i * 5);
            continue;
        }
        AStarGrid Gm = A.G;
        Gm.occ = OCC_SMEM ? s_occ : A.G.occ + (size_t)m * A.occ_words;   // (staged: the batch's one map)
        for (int w = lane; w < A.words; w += MPP_GL) vis[w] = 0u;
        grp_sync(L);
        int n = 1, cur = start, status = 1;
        if (lane == 0) { path[0] = start; vis[start >> 5] |= 1u << (start & 31); }   // pso.py:63-65
        grp_sync(L);
        for (int k = 0; k <= A.W; ++k) {
            const int goal = (k < A.W) ? A.wps[(size_t)i * A.W + k] : target;
            // the segment is written over the tail cell of the path (segment[0] == current_start)
            const int cap = A.max_cells - (n - 1);
            const int sl = astar_search(L, Gm, S, 0, cur, goal, vis, path + (n - 1), cap, nullptr, A.counters);
            if (sl < 0) { status = -1; break; }
            if (sl == 0 || (sl == 1 && cur != goal)) { status = 0; break; }          // pso.py:77,87 -> []
            if (sl > cap) { status = 2; n += sl - 1; break; }                        // truncated
            for (int t = 1 + lane; t < sl; t += MPP_GL) {                            // nodes_in_path_so_far.update
                const int c = path[n - 1 + t];
                atomicOr(&vis[c >> 5], 1u << (c & 31));
            }
            grp_sync(L);
            n += sl - 1;
            cur = goal;
        }
        // (consecutive duplicates cannot occur: a segment never repeats its first cell; pso.py:91-93 is a no-op)
        int n_out = status == 1 ? n : (status == 2 ? n : status);
        if (lane == 0) A.n_cells[i] = n_out;
        StatsCtx Xm = A.X;
        Xm.occ = Gm.occ;
        if (Xm.cls) Xm.cls += (size_t)m * rc;
        path_stats_warp(L, Xm, path, status == 1 ? n : 0, A.stats + (size_t)i * 5);
    }
}

// Waypoint chains over a batch of same-shape maps (individual i on map map_dev[i], from that map's start to its target).
extern "C" int mpp_waypoint_fitness_maps(mpp_map_batch *maps, const int32_t *map_dev, const int32_t *waypoints_dev,
                                         int n_individuals, int n_waypoints, const mpp_policy *policy, int32_t *cells_dev,
                                         int max_cells, int32_t *n_cells_dev, double *stats_dev, uint32_t *visited_dev,
                                         void *scratch_dev, size_t scratch_bytes, int n_slots, int heap_cap,
                                         unsigned long long *counters_dev, const int32_t *order_dev, void *stream) {
    MPP_REQUIRE(maps && map_dev && policy && cells_dev && n_cells_dev && stats_dev && visited_dev && scratch_dev,
                "mpp_waypoint_fitness_maps: null argument");
    MPP_REQUIRE(n_individuals > 0 && n_waypoints >= 0 && max_cells > 1, "mpp_waypoint_fitness_maps: bad sizes");
    MPP_REQUIRE(n_waypoints == 0 || waypoints_dev, "mpp_waypoint_fitness_maps: null waypoints");
    int rc = check_search(maps, scratch_bytes, n_slots, heap_cap);
    if (rc) return rc;
    MPP_CUDA(cudaSetDevice(maps->device));
    cudaStream_t s = (cudaStream_t)stream;
    ChainArgs A;
    memset(&A, 0, sizeof(A));
    rc = mpp_stats_ctx(maps, policy, stream, &A.X);
    if (rc) return rc;
    MPP_CUDA(cudaMemsetAsync(scratch_dev, 0, 256, s));
    A.G.occ = maps->occ_dev; A.G.pitch = maps->pitch_words; A.G.R = maps->rows; A.G.C = maps->cols;
    A.G.allow_diag = policy->allow_diagonal; A.G.restrict_corner = policy->restrict_policy;
    A.occ_words = maps->occ_words; A.map = map_dev; A.n_maps = maps->n_maps; A.meta = maps->meta_dev;
    A.wps = waypoints_dev; A.N = n_individuals; A.W = n_waypoints; A.words = (maps->rows * maps->cols + 31) / 32;
    A.cells = cells_dev; A.max_cells = max_cells; A.n_cells = n_cells_dev; A.stats = stats_dev; A.visited = visited_dev;
    A.scratch = (char *)scratch_dev; A.n_slots = n_slots; A.heap_cap = heap_cap; A.counters = counters_dev;
    A.order = order_dev;
    const int blocks = (n_slots + MPP_AS_GROUPS - 1) / MPP_AS_GROUPS;
    static MppStaging staging = {-1, {0}};
    bool stage;
    rc = stage_one_map((const void *)mpp_waypoint_fitness_kernel<true>, staging, maps, &stage);
    if (rc) return rc;
    if (stage) mpp_waypoint_fitness_kernel<true><<<blocks, MPP_AS_THREADS, (size_t)maps->occ_words * 4, s>>>(A);
    else mpp_waypoint_fitness_kernel<false><<<blocks, MPP_AS_THREADS, 0, s>>>(A);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}
