// mpp_mpa.cu -- one MPA iteration for the whole predator population (MPA.py:339-410): phase move
// (Brownian / Levy target generation MPA.py:250-282 + path-segment reconstruction :284-318 with the
// private A* :106-151), marine-memory saving (:380-384) and the FADs step (:387-410).
// One lane group (mpp_astar.cuh: a warp by default) per individual; every individual reads only the old (sorted) population and the elite, so
// the loop bodies of MPA.py:340/349/366/387 are data-parallel.  Streams: (seed, MPA_PHASE, it, i) and
// (seed, MPA_FADS, it, i), draws consumed in the reference's order.
#include <cmath>

#include "mpp_astar.cuh"
#include "mpp_stats.cuh"

#define MPP_MPA_THREADS (MPP_GL == 32 ? 256 : 128)
#define MPP_MPA_GROUPS (MPP_MPA_THREADS / MPP_GL)   // predators (lane groups) served by one CTA at a time
#define MPP_NV_MAGICCONST 1.7155277699214135  // random.NV_MAGICCONST = 4*exp(-0.5)/sqrt(2.0)

struct MpaArgs {
    AStarGrid G;
    int occ_words;
    StatsCtx X;
    int N, iteration, phase;          // phase 1/2/3 (MPA.py:339,348,365)
    int pred_begin, pred_end;         // predators of every map handled by this launch (a rank's shard)
    double P_const, CF, FADs_rate, levy_sigma, levy_inv_beta;
    const int32_t *cells;             // old population, sorted (or through `order`): N x max_cells
    const int32_t *n_cells;
    const double *stats;              // N x 5
    int max_cells;
    int32_t *out_cells;               // next population (unsorted): N x max_cells
    int32_t *out_n;
    double *out_stats;
    int32_t *tmp_cells;               // n_slots x max_cells
    uint32_t *avoid;                  // n_slots x words
    int words;
    char *scratch;
    int n_slots, heap_cap;
    int32_t *status;                  // [0] = worst status seen (0 ok, 1 = heap overflow, 2 = path truncated)
    unsigned long long *counters;
    // ---- batches of independent same-shape maps (blockIdx.y = map; a single map is a batch of one) ----
    const MppMapMeta *meta;           // per-map start / target
    const uint64_t *seeds;            // per-map Philox seed
    const int32_t *order;             // [n_maps][N]: predator i of the (sorted) population is row order[i] (null: identity)
    unsigned int *queue;              // [n_maps] work counters
    int warps_per_map;                // search slots serving one map
};

// CPython random.normalvariate (Kinderman-Monahan) over the stream
__device__ __forceinline__ double mpa_normalvariate(mpp_stream_rng &rng, double mu, double sigma) {
    double z;
    for (;;) {
        const double u1 = rng.draw();
        const double u2 = 1.0 - rng.draw();
        z = MPP_NV_MAGICCONST * (u1 - 0.5) / u2;
        const double zz = z * z / 4.0;
        if (zz <= -log(u2)) break;
    }
    return mu + z * sigma;
}
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// MPA.py:250-264
__device__ int mpa_levy_target(mpp_stream_rng &rng, const MpaArgs &A, int cur, double scale) {
    const int R = A.G.R, C = A.G.C;
    const double u = mpa_normalvariate(rng, 0.0, A.levy_sigma);
    double v = mpa_normalvariate(rng, 0.0, 1.0);
    if (fabs(v) < 1e-9) v = 1e-9;
    double step = 0.05 * u / pow(fabs(v), A.levy_inv_beta) * scale;
    const double lim = (double)(R > C ? R : C) * 0.5;
    step = fmin(fmax(step, -lim), lim);
    const double angle = 0.0 + (2.0 * 3.141592653589793 - 0.0) * rng.draw();
    const int dr = (int)rint(step * sin(angle)), dc = (int)rint(step * cos(angle));
    return clampi(cur / C + dr, 0, R - 1) * C + clampi(cur % C + dc, 0, C - 1);
}

// MPA.py:266-282 ; elite_node < 0 == None
__device__ int mpa_brownian_target(mpp_stream_rng &rng, const MpaArgs &A, int cur, int elite_node, double scale) {
    const int R = A.G.R, C = A.G.C;
    const int cr = cur / C, cc = cur % C;
    int tr_, tc_;
    if (rng.draw() < 0.7 && elite_node >= 0) {
        const int er = elite_node / C, ec = elite_node % C;
        const int dr = er - cr, dc = ec - cc;
        const double dist = sqrt((double)((long long)dr * dr + (long long)dc * dc));
        if (dist > 1e-6) {
            const double b = fabs(mpa_normalvariate(rng, 0.0, 1.0));
            int ms = (int)rint(scale * b * 5.0);
            if (ms < 1) ms = 1;
            const double max_step = fmin(dist, (double)ms);
            tr_ = cr + (int)rint((double)dr / dist * max_step);
            tc_ = cc + (int)rint((double)dc / dist * max_step);
        } else {
            return elite_node;
        }
    } else {
        int m = (int)rint((double)(R > C ? R : C) * 0.1 * scale * fabs(mpa_normalvariate(rng, 0.0, 1.0)));
        if (m < 1) m = 1;
        const int dr = -m + rng.below(2 * m + 1);
        const int dc = -m + rng.below(2 * m + 1);
        tr_ = cr + dr;
        tc_ = cc + dc;
    }
    return clampi(tr_, 0, R - 1) * C + clampi(tc_, 0, C - 1);
}

__device__ __forceinline__ void warp_copy_path(const LaneGroup &L, int32_t *dst, const int32_t *src, int n) {
    for (int i = L.gl; i < n; i += MPP_GL) dst[i] = src[i];
    grp_sync(L);
}
__device__ __forceinline__ void warp_mark(const LaneGroup &L, uint32_t *bits, const int32_t *cells, int n) {
    for (int i = L.gl; i < n; i += MPP_GL) atomicOr(&bits[cells[i] >> 5], 1u << (cells[i] & 31));
    grp_sync(L);
}
__device__ __forceinline__ void copy_stats(const LaneGroup &L, double *dst, const double *src) {
    if (L.gl < 5) dst[L.gl] = src[L.gl];
    grp_sync(L);
}

// MP (per-map parameters, mpp_mpa_iteration_batch_p): P_const, FADs_rate, levy_sigma, 1 / levy_beta and the statistics
// weights of params[map] replace the launch's values in this kernel's copy of A; nothing downstream changes.
template <bool OCC_SMEM, bool MP>
__global__ void __launch_bounds__(MPP_MPA_THREADS, 3)
mpp_mpa_iteration_kernel(MpaArgs A, const mpp_pop_params *__restrict__ params) {
    extern __shared__ __align__(16) uint32_t s_occ[];
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ __align__(16) uint8_t s_cnt[MPP_MPA_GROUPS][MPP_PQ_NB];
    AStarGrid G = A.G;
    StatsCtx X = A.X;
    if constexpr (MP) {
        const mpp_pop_params &P = params[blockIdx.y];
        A.P_const = P.P_const; A.FADs_rate = P.FADs_rate; A.levy_sigma = P.levy_sigma;
        A.levy_inv_beta = __ddiv_rn(1.0, P.levy_beta);
        mpp_pop_weights(X.pol, P);
    }
    if (OCC_SMEM) {
        mpp_stage_bulk(s_occ, A.G.occ + (size_t)blockIdx.y * A.occ_words, (uint32_t)A.occ_words * 4u, &s_bar);
        G.occ = s_occ;
        X.occ = s_occ;
    } else {
        G.occ = A.G.occ + (size_t)blockIdx.y * A.occ_words;
        X.occ = G.occ;
    }
    const LaneGroup L = lane_group();
    const int lane = L.gl;
    const int map = blockIdx.y;
    const int slot_in_map = (blockIdx.x * MPP_MPA_THREADS + threadIdx.x) / MPP_GL;
    if (slot_in_map >= A.warps_per_map) return;
    const int slot = map * A.warps_per_map + slot_in_map;
    const int rc = G.R * G.C, C = G.C;
    AStarSlot S = astar_slot_at(A.scratch + 256 + (size_t)slot * astar_slot_bytes(rc, A.heap_cap), rc, A.heap_cap,
                                s_cnt[threadIdx.x / MPP_GL]);
    unsigned int *next = A.queue + map;
    uint32_t *avoid = A.avoid + (size_t)slot * A.words;
    int32_t *tmp = A.tmp_cells + (size_t)slot * A.max_cells;
    const int start = A.meta[map].start, target = A.meta[map].target;
    const uint64_t seed = A.seeds[map];
    {   // this map's slice of the population buffers
        const size_t pm = (size_t)map * A.N;
        A.cells += pm * A.max_cells; A.n_cells += pm; A.stats += pm * 5;
        A.out_cells += pm * A.max_cells; A.out_n += pm; A.out_stats += pm * 5;
        if (A.order) A.order += pm;
    }
    for (;;) {
        int i = 0;
        if (lane == 0) i = A.pred_begin + (int)atomicAdd(next, 1u);
        i = grp_shfl(L, i, 0);
        if (i >= A.pred_end) break;
        int st_flag = 0;
        const int row_i = A.order ? A.order[i] : i, row_0 = A.order ? A.order[0] : 0;   // rows of predator i / the elite
        const int32_t *old_path = A.cells + (size_t)row_i * A.max_cells;
        const int old_n = A.n_cells[row_i];
        const double *old_stats = A.stats + (size_t)row_i * 5;
        const double old_fit = old_stats[4];
        const int32_t *elite_path = A.cells + (size_t)row_0 * A.max_cells;   // population[0] after the sort (MPA.py:333-334)
        const int elite_n = A.n_cells[row_0];
        const double *elite_stats = A.stats + (size_t)row_0 * 5;
        int32_t *out = A.out_cells + (size_t)i * A.max_cells;
        double *ostats = A.out_stats + (size_t)i * 5;
        // ---------------- phase move (MPA.py:339-377) ----------------
        const int32_t *P;    // path_to_modify
        const double *Pstats;
        int nP;
        const int32_t *ref;  // the path Brownian moves sample from
        int nref;
        bool levy;
        double scale, gate_p;
        if (A.phase == 1) {
            P = old_path; nP = old_n; Pstats = old_stats; ref = elite_path; nref = elite_n; levy = false;
            scale = A.P_const; gate_p = A.P_const;
        } else if (A.phase == 2) {
            levy = i < A.N / 2;
            P = levy ? old_path : elite_path; nP = levy ? old_n : elite_n; Pstats = levy ? old_stats : elite_stats;
            ref = levy ? elite_path : old_path; nref = levy ? elite_n : old_n;
            scale = levy ? A.P_const : A.P_const * A.CF; gate_p = scale;
        } else {
            P = elite_path; nP = elite_n; Pstats = elite_stats; ref = old_path; nref = old_n; levy = true;
            scale = A.P_const * A.CF; gate_p = scale;
        }
        int n_new = nP;            // candidate defaults to path_to_modify with its stats
        bool rebuilt = false;
        mpp_stream_rng rng;
        rng.init(seed, MPP_CLS_MPA_PHASE, (uint32_t)A.iteration, (uint32_t)i);
        if (nP > 1) {
            const int idx = rng.below(nP - 1);                                     // randint(0, len-2)
            if (rng.draw() < gate_p) {
                // ---- _reconstruct_path_segment MPA.py:284-318 ----
                const int cur = P[idx];
                for (int w = lane; w < A.words; w += MPP_GL) avoid[w] = 0u;
                grp_sync(L);
                warp_mark(L, avoid, P, idx);                                          // set(prefix[:-1])
                warp_copy_path(L, out, P, idx + 1);                                   // prefix
                int n = idx + 1;
                int inter;
                if (levy) inter = mpa_levy_target(rng, A, cur, scale);
                else {
                    const int elite_node = nref > 0 ? ref[rng.below(nref)] : -1;   // random.choice(elite_path) :294
                    inter = mpa_brownian_target(rng, A, cur, elite_node, scale);
                }
                int a_start = cur;
                if (!occ_bit(G, inter / C, inter % C) && inter != a_start) {       // :298
                    const int cap = A.max_cells - (n - 1);
                    const int sl = astar_search(L, G, S, 1, a_start, inter, avoid, out + (n - 1), cap, nullptr, A.counters);
                    if (sl < 0) st_flag = 1;
                    else if (sl > cap) st_flag = 2;
                    else if (sl > 1) {                                             // :300-305
                        warp_mark(L, avoid, out + n, sl - 1);
                        n += sl - 1;
                        a_start = inter;
                    }
                }
                if (a_start != target && st_flag == 0) {                           // :306-309
                    const int cap = A.max_cells - (n - 1);
                    const int sl = astar_search(L, G, S, 1, a_start, target, avoid, out + (n - 1), cap, nullptr, A.counters);
                    if (sl < 0) st_flag = 1;
                    else if (sl > cap) st_flag = 2;
                    else if (sl > 1) n += sl - 1;
                }
                // (consecutive duplicates cannot occur; :310-315 is a no-op)
                if (st_flag == 0 && n > 0 && out[0] == start && out[n - 1] == target) {       // :316
                    n_new = n;
                    rebuilt = true;
                    path_stats_warp(L, X, out, n, ostats);
                    grp_sync(L);
                }
            }
        }
        double cand_fit = rebuilt ? ostats[4] : Pstats[4];
        // ---------------- marine memory saving MPA.py:380-384 ----------------
        int cur_n;
        double cur_fit;
        if (cand_fit < old_fit) {
            if (!rebuilt) { warp_copy_path(L, out, P, nP < A.max_cells ? nP : A.max_cells); copy_stats(L, ostats, Pstats); }
            cur_n = n_new; cur_fit = cand_fit;
        } else {
            warp_copy_path(L, out, old_path, old_n < A.max_cells ? old_n : A.max_cells);
            copy_stats(L, ostats, old_stats);
            cur_n = old_n; cur_fit = old_fit;
        }
        // ---------------- FADs MPA.py:387-410 ----------------
        mpp_stream_rng fr;
        fr.init(seed, MPP_CLS_MPA_FADS, (uint32_t)A.iteration, (uint32_t)i);
        if (fr.draw() < A.FADs_rate && st_flag == 0) {
            int n2 = 0;
            if (fr.draw() < A.CF) {
                const int r = fr.below(G.R), c = fr.below(G.C);                    // :391
                const int node = r * C + c;
                if (!occ_bit(G, r, c)) {
                    const int sl1 = astar_search(L, G, S, 1, start, node, nullptr, tmp, A.max_cells, nullptr, A.counters);
                    if (sl1 < 0) st_flag = 1;
                    else if (sl1 > A.max_cells) st_flag = 2;
                    else if (sl1 > 0) {
                        for (int w = lane; w < A.words; w += MPP_GL) avoid[w] = 0u;
                        grp_sync(L);
                        warp_mark(L, avoid, tmp, sl1 - 1);                            // set(p1[:-1]) :396
                        const int cap = A.max_cells - (sl1 - 1);
                        const int sl2 = astar_search(L, G, S, 1, node, target, avoid, tmp + (sl1 - 1), cap, nullptr, A.counters);
                        if (sl2 < 0) st_flag = 1;
                        else if (sl2 > cap) st_flag = 2;
                        else if (sl2 > 0) {
                            const int nn = sl1 + sl2 - 1;                          // p1 + p2[1:]
                            if (tmp[nn - 1] == target) n2 = nn;                    // :400
                        }
                    }
                }
            } else {
                const int sl = astar_search(L, G, S, 1, start, target, nullptr, tmp, A.max_cells, nullptr, A.counters);  // :405
                if (sl < 0) st_flag = 1;
                else if (sl > A.max_cells) st_flag = 2;
                else if (sl > 0) n2 = sl;
            }
            if (n2 > 0 && st_flag == 0) {
                double *slot_stats = (double *)((char *)S.hdr + 64);               // 5 doubles in the slot header
                path_stats_warp(L, X, tmp, n2, slot_stats);
                grp_sync(L);
                const double f2 = slot_stats[4];
                if (f2 < cur_fit) {                                                // :402 / :408
                    warp_copy_path(L, out, tmp, n2);
                    copy_stats(L, ostats, slot_stats);
                    cur_n = n2; cur_fit = f2;
                }
            }
        }
        if (lane == 0) {
            A.out_n[i] = cur_n;
            if (st_flag) atomicMax(A.status, st_flag);
        }
        grp_sync(L);
    }
}

template <bool MP>
static int mpa_launch(MpaArgs &A, const mpp_pop_params *params_dev, int n_maps, int device, size_t occ_bytes,
                      cudaStream_t s) {
    const int blocks = (A.warps_per_map + MPP_MPA_GROUPS - 1) / MPP_MPA_GROUPS;
    const dim3 grid(blocks, n_maps);
    static MppStaging staging = {-1, {0}};
    bool stage = false;
    const int rc = mpp_occ_staging((const void *)mpp_mpa_iteration_kernel<true, MP>, staging, device, occ_bytes, &stage);
    if (rc) return rc;
    if (stage) mpp_mpa_iteration_kernel<true, MP><<<grid, MPP_MPA_THREADS, occ_bytes, s>>>(A, params_dev);
    else mpp_mpa_iteration_kernel<false, MP><<<grid, MPP_MPA_THREADS, 0, s>>>(A, params_dev);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

// ---------------------------------------------------------------------------------------------
// Batches of independent same-shape maps (BASELINE config 5; a single map is a batch of one): one launch serves the
// predators of every map (blockIdx.y = map; `warps_per_map` search slots and one work queue per map).  The population
// buffers are [n_maps][N][...]; the kernel reads the OLD population through `order` when given (the stable argsort of
// its fitness column, computed on the device by the caller), so the sorts of MPA.py:333,412 never move a path.
// ---------------------------------------------------------------------------------------------
// params_dev: per-map parameters (mpp_mpa_iteration_batch_p; the scalars are then unused) or null
static int mpa_iteration(const mpp_map_batch *maps, const mpp_policy *policy, const mpp_pop_params *params_dev,
                         int n_predators, int pred_begin, int pred_end, int iteration, int phase, double P_const,
                         double CF, double FADs_rate, double levy_sigma, double levy_beta, const uint64_t *seeds_dev,
                         const int32_t *order_dev, const int32_t *cells_dev, const int32_t *n_cells_dev,
                         const double *stats_dev, int max_cells, int32_t *out_cells_dev, int32_t *out_n_dev,
                         double *out_stats_dev, int32_t *tmp_cells_dev, uint32_t *avoid_dev, void *scratch_dev,
                         size_t scratch_bytes, int warps_per_map, int heap_cap, uint32_t *queue_dev, int32_t *status_dev,
                         unsigned long long *counters_dev, void *stream, const char *who) {
    MPP_REQUIRE(maps && policy && seeds_dev && cells_dev && n_cells_dev && stats_dev && out_cells_dev &&
                    out_n_dev && out_stats_dev && tmp_cells_dev && avoid_dev && scratch_dev && queue_dev && status_dev,
                "%s: null argument", who);
    MPP_REQUIRE(n_predators > 0 && max_cells > 1 && phase >= 1 && phase <= 3 && warps_per_map > 0 && heap_cap >= 64,
                "%s: bad sizes", who);
    MPP_REQUIRE(pred_begin >= 0 && pred_begin <= pred_end && pred_end <= n_predators, "%s: bad predator range", who);
    if (pred_begin == pred_end) return MPP_OK;
    MPP_REQUIRE(maps->rows < 32768 && maps->cols < 65536, "%s: map exceeds the packed-node limit", who);
    const int rc = maps->rows * maps->cols;
    const size_t need = 256 + (size_t)warps_per_map * maps->n_maps * astar_slot_bytes(rc, heap_cap);
    MPP_REQUIRE(scratch_bytes >= need, "%s: scratch too small (%zu < %zu)", who, scratch_bytes, need);
    for (int k = 0; k < maps->n_maps; ++k)
        MPP_REQUIRE(maps->meta_host[k].start >= 0 && maps->meta_host[k].target >= 0, "%s: map %d has no start/target", who, k);
    MPP_CUDA(cudaSetDevice(maps->device));
    cudaStream_t s = (cudaStream_t)stream;
    MpaArgs A;
    mpp_policy pol = *policy;
    pol.mode = 1;                                                      // MPA.py:164-173: safety = 0.0
    int err = mpp_stats_ctx(const_cast<mpp_map_batch *>(maps), &pol, stream, &A.X);   // (mode 1 builds no tables)
    if (err) return err;
    MPP_CUDA(cudaMemsetAsync(queue_dev, 0, sizeof(uint32_t) * maps->n_maps, s));
    A.G.occ = maps->occ_dev; A.G.pitch = maps->pitch_words; A.G.R = maps->rows; A.G.C = maps->cols;
    A.G.allow_diag = policy->allow_diagonal; A.G.restrict_corner = policy->restrict_policy;
    A.occ_words = maps->occ_words;
    A.N = n_predators; A.iteration = iteration; A.phase = phase;
    A.pred_begin = pred_begin; A.pred_end = pred_end;
    A.P_const = P_const; A.CF = CF; A.FADs_rate = FADs_rate; A.levy_sigma = levy_sigma; A.levy_inv_beta = 1.0 / levy_beta;
    A.cells = cells_dev; A.n_cells = n_cells_dev; A.stats = stats_dev; A.max_cells = max_cells;
    A.out_cells = out_cells_dev; A.out_n = out_n_dev; A.out_stats = out_stats_dev;
    A.tmp_cells = tmp_cells_dev; A.avoid = avoid_dev; A.words = (rc + 31) / 32;
    A.scratch = (char *)scratch_dev; A.n_slots = warps_per_map * maps->n_maps; A.heap_cap = heap_cap; A.status = status_dev;
    A.counters = counters_dev;
    A.meta = maps->meta_dev; A.seeds = seeds_dev; A.order = order_dev; A.queue = queue_dev; A.warps_per_map = warps_per_map;
    const size_t occ_bytes = (size_t)maps->occ_words * 4;
    return params_dev ? mpa_launch<true>(A, params_dev, maps->n_maps, maps->device, occ_bytes, s)
                      : mpa_launch<false>(A, nullptr, maps->n_maps, maps->device, occ_bytes, s);
}

extern "C" int mpp_mpa_iteration_batch(const mpp_map_batch *maps, const mpp_policy *policy, int n_predators,
                                       int pred_begin, int pred_end, int iteration, int phase, double P_const, double CF, double FADs_rate, double levy_sigma,
                                       double levy_beta, const uint64_t *seeds_dev, const int32_t *order_dev,
                                       const int32_t *cells_dev, const int32_t *n_cells_dev, const double *stats_dev,
                                       int max_cells, int32_t *out_cells_dev, int32_t *out_n_dev, double *out_stats_dev,
                                       int32_t *tmp_cells_dev, uint32_t *avoid_dev, void *scratch_dev, size_t scratch_bytes,
                                       int warps_per_map, int heap_cap, uint32_t *queue_dev, int32_t *status_dev,
                                       unsigned long long *counters_dev, void *stream) {
    return mpa_iteration(maps, policy, nullptr, n_predators, pred_begin, pred_end, iteration, phase, P_const, CF,
                         FADs_rate, levy_sigma, levy_beta, seeds_dev, order_dev, cells_dev, n_cells_dev, stats_dev,
                         max_cells, out_cells_dev, out_n_dev, out_stats_dev, tmp_cells_dev, avoid_dev, scratch_dev,
                         scratch_bytes, warps_per_map, heap_cap, queue_dev, status_dev, counters_dev, stream,
                         "mpp_mpa_iteration_batch");
}

extern "C" int mpp_mpa_iteration_batch_p(const mpp_map_batch *maps, const mpp_policy *policy, int n_predators,
                                         int pred_begin, int pred_end, int iteration, int phase,
                                         const mpp_pop_params *params_dev, double CF, const uint64_t *seeds_dev,
                                         const int32_t *order_dev, const int32_t *cells_dev, const int32_t *n_cells_dev,
                                         const double *stats_dev, int max_cells, int32_t *out_cells_dev,
                                         int32_t *out_n_dev, double *out_stats_dev, int32_t *tmp_cells_dev,
                                         uint32_t *avoid_dev, void *scratch_dev, size_t scratch_bytes,
                                         int warps_per_map, int heap_cap, uint32_t *queue_dev, int32_t *status_dev,
                                         unsigned long long *counters_dev, void *stream) {
    MPP_REQUIRE(params_dev, "mpp_mpa_iteration_batch_p: null params_dev");
    return mpa_iteration(maps, policy, params_dev, n_predators, pred_begin, pred_end, iteration, phase, 0.0, CF, 0.0,
                         0.0, 1.0, seeds_dev, order_dev, cells_dev, n_cells_dev, stats_dev, max_cells, out_cells_dev,
                         out_n_dev, out_stats_dev, tmp_cells_dev, avoid_dev, scratch_dev, scratch_bytes, warps_per_map,
                         heap_cap, queue_dev, status_dev, counters_dev, stream, "mpp_mpa_iteration_batch_p");
}

// The initial population of every map (MPA.py:231-245): N identical runs of the private A* start -> target are ONE
// search per map; row 0 of each map's buffers receives the path ([start, target] when there is none, :236) and its
// statistics -- the caller replicates the row.  One warp per map.
// MP (mpp_mpa_init_batch_p): the statistics weights of params[map] in place of A.X.pol's
template <bool MP>
__global__ void __launch_bounds__(MPP_MPA_THREADS)
mpp_mpa_init_kernel(MpaArgs A, int n_maps, const mpp_pop_params *__restrict__ params) {
    __shared__ __align__(16) uint8_t s_cnt[MPP_MPA_GROUPS][MPP_PQ_NB];
    const LaneGroup L = lane_group();
    const int lane = L.gl;
    const int map = (blockIdx.x * MPP_MPA_THREADS + threadIdx.x) / MPP_GL;
    if (map >= n_maps) return;
    AStarGrid G = A.G;
    StatsCtx X = A.X;
    G.occ = A.G.occ + (size_t)map * A.occ_words;
    X.occ = G.occ;
    const int rc = G.R * G.C;
    AStarSlot S = astar_slot_at(A.scratch + 256 + (size_t)map * astar_slot_bytes(rc, A.heap_cap), rc, A.heap_cap,
                                s_cnt[threadIdx.x / MPP_GL]);
    const int start = A.meta[map].start, target = A.meta[map].target;
    int32_t *out = A.out_cells + (size_t)map * A.N * A.max_cells;
    int sl = astar_search(L, G, S, 1, start, target, nullptr, out, A.max_cells, nullptr, A.counters);
    int st_flag = 0;
    if (sl < 0) { st_flag = 1; sl = 0; }
    else if (sl > A.max_cells) { st_flag = 2; sl = 0; }
    if (sl == 0) {                                                     // :236 (the target cell is never an obstacle)
        if (lane == 0) { out[0] = start; out[1] = target; }
        sl = 2;
        grp_sync(L);
    }
    if constexpr (MP) mpp_pop_weights(X.pol, params[map]);         // (loaded after the search: not live across it)
    path_stats_warp(L, X, out, sl, A.out_stats + (size_t)map * A.N * 5);
    if (lane == 0) {
        A.out_n[(size_t)map * A.N] = sl;
        if (st_flag) atomicMax(A.status, st_flag);
    }
}

static int mpa_init(const mpp_map_batch *maps, const mpp_policy *policy, const mpp_pop_params *params_dev,
                    int n_predators, int max_cells, int32_t *cells_dev, int32_t *n_cells_dev, double *stats_dev,
                    void *scratch_dev, size_t scratch_bytes, int heap_cap, int32_t *status_dev,
                    unsigned long long *counters_dev, void *stream, const char *who) {
    MPP_REQUIRE(maps && policy && cells_dev && n_cells_dev && stats_dev && scratch_dev && status_dev,
                "%s: null argument", who);
    MPP_REQUIRE(n_predators > 0 && max_cells > 1 && heap_cap >= 64, "%s: bad sizes", who);
    MPP_REQUIRE(maps->rows < 32768 && maps->cols < 65536, "%s: map exceeds the packed-node limit", who);
    const int rc = maps->rows * maps->cols;
    MPP_REQUIRE(scratch_bytes >= 256 + (size_t)maps->n_maps * astar_slot_bytes(rc, heap_cap), "%s: scratch too small", who);
    for (int k = 0; k < maps->n_maps; ++k)
        MPP_REQUIRE(maps->meta_host[k].start >= 0 && maps->meta_host[k].target >= 0, "%s: map %d has no start/target", who, k);
    MPP_CUDA(cudaSetDevice(maps->device));
    MpaArgs A;
    memset(&A, 0, sizeof(A));
    mpp_policy pol = *policy;
    pol.mode = 1;                                                      // MPA.py:164-173: safety = 0.0
    const int err = mpp_stats_ctx(const_cast<mpp_map_batch *>(maps), &pol, stream, &A.X);   // (mode 1 builds no tables)
    if (err) return err;
    A.G.occ = maps->occ_dev; A.G.pitch = maps->pitch_words; A.G.R = maps->rows; A.G.C = maps->cols;
    A.G.allow_diag = policy->allow_diagonal; A.G.restrict_corner = policy->restrict_policy;
    A.occ_words = maps->occ_words; A.N = n_predators; A.max_cells = max_cells;
    A.out_cells = cells_dev; A.out_n = n_cells_dev; A.out_stats = stats_dev;
    A.scratch = (char *)scratch_dev; A.heap_cap = heap_cap; A.status = status_dev; A.counters = counters_dev;
    A.meta = maps->meta_dev;
    const int blocks = (maps->n_maps + MPP_MPA_GROUPS - 1) / MPP_MPA_GROUPS;
    if (params_dev)
        mpp_mpa_init_kernel<true><<<blocks, MPP_MPA_THREADS, 0, (cudaStream_t)stream>>>(A, maps->n_maps, params_dev);
    else mpp_mpa_init_kernel<false><<<blocks, MPP_MPA_THREADS, 0, (cudaStream_t)stream>>>(A, maps->n_maps, nullptr);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

extern "C" int mpp_mpa_init_batch(const mpp_map_batch *maps, const mpp_policy *policy, int n_predators, int max_cells,
                                  int32_t *cells_dev, int32_t *n_cells_dev, double *stats_dev, void *scratch_dev,
                                  size_t scratch_bytes, int heap_cap, int32_t *status_dev, unsigned long long *counters_dev,
                                  void *stream) {
    return mpa_init(maps, policy, nullptr, n_predators, max_cells, cells_dev, n_cells_dev, stats_dev, scratch_dev,
                    scratch_bytes, heap_cap, status_dev, counters_dev, stream, "mpp_mpa_init_batch");
}

extern "C" int mpp_mpa_init_batch_p(const mpp_map_batch *maps, const mpp_policy *policy, const mpp_pop_params *params_dev,
                                    int n_predators, int max_cells, int32_t *cells_dev, int32_t *n_cells_dev,
                                    double *stats_dev, void *scratch_dev, size_t scratch_bytes, int heap_cap,
                                    int32_t *status_dev, unsigned long long *counters_dev, void *stream) {
    MPP_REQUIRE(params_dev, "mpp_mpa_init_batch_p: null params_dev");
    return mpa_init(maps, policy, params_dev, n_predators, max_cells, cells_dev, n_cells_dev, stats_dev, scratch_dev,
                    scratch_bytes, heap_cap, status_dev, counters_dev, stream, "mpp_mpa_init_batch_p");
}
