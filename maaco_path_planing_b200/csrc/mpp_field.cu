// mpp_field.cu -- exact Dijkstra distance fields: g* and the parent move of every cell of a map, from one source, and
// the reference's path to any target read from them.
// Reference semantics: dijkstra.py:32-97 (= mpp_astar.cuh variant 2: extract-min over (g, r, c), strict relaxation,
// closed set, stop at the target).
//
// Why a field reproduces the reference bit for bit:
//   * fp64 addition rounds monotonically and every step weighs w >= 1 (1 or sqrt 2), so fl(g + w) > g.  The g with
//     which the reference pops a cell is the least fixed point g*(n) = min over allowed neighbours p of
//     fl(g*(p) + w(p, n)), g*(src) = 0 -- whatever order the relaxations come in.
//   * Buckets of width 1 settle in one sweep: a cell of bucket k = floor(g*) has every minimising predecessor in a bucket
//     < k (fl(g_p + 1) >= k + 1 when g_p >= k), and a cell of bucket k relaxes only into k+1 and k+2.  So the buckets are
//     swept in order, each once.  The relaxations are 64-bit atomicMin on the g bit patterns: positive doubles and +inf
//     order like unsigned integers, so the order of the atomics cannot change the result.
//   * The reference keeps the FIRST strict improvement to the final value, and pops in (g, cell) order: parent(n) is the
//     allowed neighbour p with fl(g*(p) + w) == g*(n) and the least (g*(p), cell p) -- a per-cell pass over the finished
//     field.
// (A* is another matter: with a floating-point heuristic it can pop a cell one ulp above g*, so it has no field form.)
#include <cooperative_groups.h>

#include "mpp_astar.cuh"
#include "mpp_stats.cuh"

namespace cg = cooperative_groups;

#define MPP_FIELD_THREADS 512
#define MPP_FIELD_PATH_THREADS 256
#define MPP_FIELD_UNLISTED 0x7fffffff

// per-map scratch: [0,256) bucket counts (a ring of 4), listed[rc] (least bucket the cell was listed in), then the ring
// of three bucket lists of rc cells each
static __host__ __device__ __forceinline__ size_t field_list_words(int rc) { return astar_align256((size_t)rc * 4) / 4; }
static __host__ __device__ __forceinline__ size_t field_scratch_bytes(int rc) {
    return 256 + 4 * field_list_words(rc) * 4;
}

struct FieldArgs {
    AStarGrid G;            // G.occ: map 0's occupancy
    int occ_words;
    int cs;                 // CTAs per map (the cluster)
    const int32_t *src;     // [n_maps]
    double *g;              // [n_maps][rc]
    uint8_t *parent;        // [n_maps][rc]
    char *scratch;          // [n_maps][field_scratch_bytes(rc)]
};

// One cluster of A.cs CTAs per map.  Sweep k reads the list of bucket k (slot k % 3), relaxes every (cell, move) pair of
// it with one thread each and appends the cells it lowers into buckets k+1 / k+2 (slots (k+1) % 3, (k+2) % 3); the
// cluster barrier separates the sweeps.  A cell is listed in a bucket at most once (atomicMin on its listed word: a
// cell's buckets only go down); an entry whose cell has since dropped into a lower bucket is stale and skipped.  The
// counts live in a ring of four: count (k+3) % 4 is neither read nor appended to during sweep k, so it is reset then.
__global__ void __launch_bounds__(MPP_FIELD_THREADS) mpp_dijkstra_field_kernel(FieldArgs A) {
    cg::cluster_group cluster = cg::this_cluster();
    const int m = blockIdx.x / A.cs;
    const int tid = (blockIdx.x % A.cs) * MPP_FIELD_THREADS + threadIdx.x, nth = A.cs * MPP_FIELD_THREADS;
    AStarGrid G = A.G;
    G.occ += (size_t)m * A.occ_words;
    const int C = G.C, rc = G.R * C;
    double *g = A.g + (size_t)m * rc;
    unsigned long long *gbits = reinterpret_cast<unsigned long long *>(g);
    uint8_t *par = A.parent + (size_t)m * rc;
    char *base = A.scratch + (size_t)m * field_scratch_bytes(rc);
    int *cnt = reinterpret_cast<int *>(base);
    int *listed = reinterpret_cast<int *>(base + 256);
    const size_t lw = field_list_words(rc);
    int *lists = listed + lw;
    const int src = A.src[m];
    const bool ok = (unsigned)src < (unsigned)rc && !occ_bit(G, src / C, src % C);   // else: an all-inf field
    for (int i = tid; i < rc; i += nth) {
        const bool s = ok && i == src;
        gbits[i] = s ? 0ull : (unsigned long long)MPP_INF_BITS;
        par[i] = 0xFF;
        listed[i] = s ? 0 : MPP_FIELD_UNLISTED;
    }
    if (tid == 0) {
        cnt[0] = ok ? 1 : 0; cnt[1] = 0; cnt[2] = 0; cnt[3] = 0;
        if (ok) lists[0] = src;
    }
    cluster.sync();
    if (!ok) return;
    const int sh = G.allow_diag ? 3 : 2;                     // moves per cell: 1 << sh
    for (int k = 0;; ++k) {
        const int n = __ldcg(&cnt[k & 3]);
        const int *lst = lists + (size_t)(k % 3) * lw;
        if (tid == 0) cnt[(k + 3) & 3] = 0;
        for (int i = tid; i < (n << sh); i += nth) {
            const int u = __ldcg(&lst[i >> sh]);
            const double gu = __ldcg(&g[u]);
            if ((int)gu != k) continue;                      // stale: the cell settled in a lower bucket
            const int mv = i & ((1 << sh) - 1);
            const int ur = u / C, uc = u % C;
            const int vr = ur + (int)((MPP_NB_R >> (2 * mv)) & 3u) - 1, vc = uc + (int)((MPP_NB_C >> (2 * mv)) & 3u) - 1;
            if (occ_bit(G, vr, vc)) continue;                // helper.py:14-16 (border = blocked)
            if (mv >= 4 && G.restrict_corner && (occ_bit(G, vr, uc) || occ_bit(G, ur, vc))) continue;   // helper.py:45-49
            const double tg = gu + (mv >= 4 ? MPP_ASTAR_SQRT2 : 1.0);
            const int v = vr * C + vc;
            if (!(tg < __ldcg(&g[v]))) continue;
            const unsigned long long tb = (unsigned long long)__double_as_longlong(tg);
            if (atomicMin(&gbits[v], tb) <= tb) continue;
            const int b = (int)tg;
            if (atomicMin(&listed[v], b) <= b) continue;     // already listed in this bucket (or a lower one)
            const int pos = atomicAdd(&cnt[b & 3], 1);
            lists[(size_t)(b % 3) * lw + pos] = v;
        }
        cluster.sync();
        if (__ldcg(&cnt[(k + 1) & 3]) == 0 && __ldcg(&cnt[(k + 2) & 3]) == 0) break;   // (uniform: both are final here)
    }
    // parent pass over the finished field
    const double INF = __longlong_as_double(MPP_INF_BITS);
    for (int v = tid; v < rc; v += nth) {
        const double gv = __ldcg(&g[v]);
        if (!(gv < INF)) continue;                           // obstacle or unreachable
        const int vr = v / C, vc = v % C;
        double bg = INF;
        int bp = 0x7fffffff, bm = 0xFF;
        for (int mv = 0; mv < (1 << sh); ++mv) {
            const int pr = vr + (int)((MPP_NB_R >> (2 * mv)) & 3u) - 1, pc = vc + (int)((MPP_NB_C >> (2 * mv)) & 3u) - 1;
            if (occ_bit(G, pr, pc)) continue;
            if (mv >= 4 && G.restrict_corner && (occ_bit(G, pr, vc) || occ_bit(G, vr, pc))) continue;   // symmetric
            const double gp = __ldcg(&g[pr * C + pc]);
            if (!(gp + (mv >= 4 ? MPP_ASTAR_SQRT2 : 1.0) == gv)) continue;
            const int p = pr * C + pc;
            if (gp < bg || (gp == bg && p < bp)) { bg = gp; bp = p; bm = mv < 4 ? (mv ^ 1) : 11 - mv; }   // move p -> v
        }
        par[v] = (uint8_t)bm;                                // the source keeps 0xFF (no p has g + w == 0)
    }
}

extern "C" size_t mpp_dijkstra_field_scratch_bytes(const mpp_map_batch *maps) {
    if (!maps) return 0;
    return (size_t)maps->n_maps * field_scratch_bytes(maps->rows * maps->cols);
}

// CTAs per map: a power of two up to 16 with n_maps * cs <= SMs (16 needs the non-portable cluster size, used when the
// device can schedule such a cluster of this kernel); a batch of about one map per SM or more runs one CTA per map.
static int field_cluster_size(const mpp_map_batch *maps, int *cs) {
    static int allow16[64];                                  // per device: 0 unknown, 1 yes, 2 no
    int c = 1;
    while (c < 16 && (long long)maps->n_maps * c * 2 <= maps->sm_count) c *= 2;
    if (c == 16) {
        int &a = allow16[maps->device & 63];
        if (a == 0) {
            a = 2;
            if (cudaFuncSetAttribute(mpp_dijkstra_field_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) ==
                cudaSuccess) {
                cudaLaunchConfig_t cfg = {};
                cudaLaunchAttribute at[1];
                at[0].id = cudaLaunchAttributeClusterDimension;
                at[0].val.clusterDim.x = 16; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
                cfg.gridDim = dim3(16); cfg.blockDim = dim3(MPP_FIELD_THREADS); cfg.attrs = at; cfg.numAttrs = 1;
                int n = 0;
                if (cudaOccupancyMaxActiveClusters(&n, mpp_dijkstra_field_kernel, &cfg) == cudaSuccess && n > 0) a = 1;
            }
            cudaGetLastError();                              // a refused attribute is not an error of this call
        }
        if (a != 1) c = 8;
    }
    *cs = c;
    return MPP_OK;
}

extern "C" int mpp_dijkstra_fields(const mpp_map_batch *maps, const int32_t *src_dev, int allow_diagonal,
                                   int restrict_corner, double *g_dev, uint8_t *parent_dev, void *scratch_dev,
                                   size_t scratch_bytes, void *stream) {
    MPP_REQUIRE(maps && src_dev && g_dev && parent_dev && scratch_dev, "mpp_dijkstra_fields: null argument");
    MPP_REQUIRE((long long)maps->rows * maps->cols < (1ll << 28), "mpp_dijkstra_fields: map %dx%d has 2^28 cells or more",
                maps->rows, maps->cols);
    MPP_REQUIRE(scratch_bytes >= mpp_dijkstra_field_scratch_bytes(maps), "mpp_dijkstra_fields: scratch too small (%zu < %zu)",
                scratch_bytes, mpp_dijkstra_field_scratch_bytes(maps));
    MPP_CUDA(cudaSetDevice(maps->device));
    int cs = 1;
    int rc = field_cluster_size(maps, &cs);
    if (rc) return rc;
    FieldArgs A;
    A.G.occ = maps->occ_dev; A.G.pitch = maps->pitch_words; A.G.R = maps->rows; A.G.C = maps->cols;
    A.G.allow_diag = allow_diagonal ? 1 : 0; A.G.restrict_corner = restrict_corner ? 1 : 0;
    A.occ_words = maps->occ_words; A.cs = cs; A.src = src_dev; A.g = g_dev; A.parent = parent_dev;
    A.scratch = (char *)scratch_dev;
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3((unsigned)maps->n_maps * cs);
    cfg.blockDim = dim3(MPP_FIELD_THREADS);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = (cudaStream_t)stream;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    MPP_CUDA(cudaLaunchKernelEx(&cfg, mpp_dijkstra_field_kernel, A));
    return MPP_OK;
}

struct FieldPathArgs {
    int C, rc, n_maps, n;
    const double *g;
    const uint8_t *parent;
    const int32_t *map, *dst;
    int32_t *cells;
    int max_cells;
    int32_t *n_cells;
    double *g_out;
    int occ_words;
    StatsCtx X;             // X.occ: map 0's occupancy, X.cls: [n_maps][rc] classes or null
    double *stats;          // n x 5 or null
};

// One lane group per query: the parent chain dst -> source, written forward, and (with A.stats) its statistics.
__global__ void __launch_bounds__(MPP_FIELD_PATH_THREADS) mpp_dijkstra_field_paths_kernel(FieldPathArgs A) {
    const LaneGroup L = lane_group();
    const int i = (blockIdx.x * MPP_FIELD_PATH_THREADS + threadIdx.x) / MPP_GL;
    if (i >= A.n) return;
    const int m = A.map[i], dst = A.dst[i];
    const double INF = __longlong_as_double(MPP_INF_BITS);
    int32_t *path = A.cells + (size_t)i * A.max_cells;
    double gd = INF;
    int len = 0;
    if ((unsigned)m < (unsigned)A.n_maps && (unsigned)dst < (unsigned)A.rc) gd = A.g[(size_t)m * A.rc + dst];
    if (gd < INF) {                                          // dijkstra.py:64-70
        if (L.gl == 0) {
            const uint8_t *pm = A.parent + (size_t)m * A.rc;
            int t = dst;
            for (;;) {
                if (len < A.max_cells) path[len] = t;
                ++len;
                const uint32_t mv = pm[t];
                if (mv == 0xFFu) break;                      // the source
                t -= ((int)((MPP_NB_R >> (2 * mv)) & 3u) - 1) * A.C + (int)((MPP_NB_C >> (2 * mv)) & 3u) - 1;
            }
        }
        len = grp_shfl(L, len, 0);
        grp_sync(L);
        const int k = len < A.max_cells ? len : A.max_cells;   // (truncated: the caller sees len > max_cells)
        for (int j = L.gl; j < k / 2; j += MPP_GL) {
            const int32_t a = path[j], b = path[k - 1 - j];
            path[j] = b; path[k - 1 - j] = a;
        }
        grp_sync(L);
    } else {
        gd = INF;
    }
    if (L.gl == 0) { A.n_cells[i] = len; if (A.g_out) A.g_out[i] = gd; }
    if (A.stats) {                                           // helper.py:98-113
        StatsCtx X = A.X;
        const int mm = (unsigned)m < (unsigned)A.n_maps ? m : 0;
        X.occ += (size_t)mm * A.occ_words;
        if (X.cls) X.cls += (size_t)mm * A.rc;
        path_stats_warp(L, X, path, (len > 0 && len <= A.max_cells) ? len : 0, A.stats + (size_t)i * 5);
    }
}

extern "C" int mpp_dijkstra_field_paths(mpp_map_batch *maps, const double *g_dev, const uint8_t *parent_dev,
                                        const int32_t *map_dev, const int32_t *dst_dev, int n,
                                        const mpp_policy *stats_policy, int32_t *cells_dev, int max_cells,
                                        int32_t *n_cells_dev, double *g_out_dev, double *stats_dev, void *stream) {
    MPP_REQUIRE(maps && g_dev && parent_dev && map_dev && dst_dev && cells_dev && n_cells_dev,
                "mpp_dijkstra_field_paths: null argument");
    MPP_REQUIRE(!stats_policy || stats_dev, "mpp_dijkstra_field_paths: stats_policy without stats_dev");
    MPP_REQUIRE(n > 0 && max_cells > 0, "mpp_dijkstra_field_paths: bad sizes");
    MPP_CUDA(cudaSetDevice(maps->device));
    FieldPathArgs A;
    memset(&A, 0, sizeof(A));
    if (stats_policy) {
        const int rc = mpp_stats_ctx(maps, stats_policy, stream, &A.X);
        if (rc) return rc;
        A.stats = stats_dev;
    }
    A.C = maps->cols; A.rc = maps->rows * maps->cols; A.n_maps = maps->n_maps; A.n = n;
    A.g = g_dev; A.parent = parent_dev; A.map = map_dev; A.dst = dst_dev;
    A.cells = cells_dev; A.max_cells = max_cells; A.n_cells = n_cells_dev; A.g_out = g_out_dev;
    A.occ_words = maps->occ_words;
    const int per_block = MPP_FIELD_PATH_THREADS / MPP_GL;
    mpp_dijkstra_field_paths_kernel<<<(n + per_block - 1) / per_block, MPP_FIELD_PATH_THREADS, 0, (cudaStream_t)stream>>>(A);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}
