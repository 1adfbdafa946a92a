// mpp_maaco.cu -- MAACO colony pass on B200: per-pass move ranking, tour construction (one thread per ant),
// order-dependent best tracking, and the atomics-free ordered pheromone update -- every kernel batched over
// independent same-shape maps (blockIdx.y = map; a single map is a batch of one).
// Reference semantics: MAACO.py:58-91 (tables), :100-181 (filter), :197-262 (selection),
// :278-302 (tour), :304-332 (pheromone), :343-358 (best tracking).
//
// Data layout of one colony (n_ants ants on an R x C map; TR x TC tiles of 32 x 32 cells):
//   slabs    [tile][ant][32] uint32   the visited bits of `ant` inside `tile`, one word per tile row -- written by the
//                                     tour kernel as whole 128-byte lines when a tile leaves the ant's shared-memory
//                                     window, read back (rarely) when the ant re-enters a tile, and streamed by the
//                                     pheromone update, which only ever touches the (tile, ant) pairs that exist
//   touched  [2][tile][ceil(n_ants/32)] uint32  bit = (tile, ant) has a slab this pass; double buffered by pass parity
//                                     (the update of pass p clears the buffer pass p+1 will use)
//   moves    [ant][max_cells] uint8   the tour as move codes (MAACO.py:98 order): the best path is decoded from them,
//                                     and they are what a sharded colony exchanges when it has no peer access
#include <type_traits>
#include <algorithm>
#include <cmath>
#include <exception>
#include <cstdlib>
#include <thread>
#include <vector>

#include "mpp_common.cuh"
#include "mpp_libm.cuh"

// ---------------------------------------------------------------------------------------------
// host: tables (libm exp/pow == what CPython / NumPy call, so the tables are bit-identical)
// ---------------------------------------------------------------------------------------------
static inline double hdist(int r0, int c0, int r1, int c1) {
    long long dr = r0 - r1, dc = c0 - c1;
    return std::sqrt((double)(dr * dr + dc * dc));
}

extern "C" double mpp_maaco_q0(int K, int k, double q0_initial) {  // MAACO.py:212-226
    double k0 = 0.7 * (double)K, q0;
    if ((double)k < k0) {
        if (std::fabs((double)K - k0) < 1e-6) q0 = q0_initial;
        else q0 = ((double)(K - k) / (double)K) * q0_initial;
    } else {
        double q0_at_k0 = (((double)K - k0) / (double)K) * q0_initial;
        q0 = q0_at_k0 +
             (((double)k - k0) / ((double)K - k0 + 1e-9)) * (q0_initial * (1 - ((double)K - k0) / (double)K) / 2.0);
    }
    q0 = q0 > 0.01 ? q0 : 0.01;
    return q0 < 0.99 ? q0 : 0.99;
}

// Rows [r_lo, r_hi) of the tables of an R x C map with the given start / target: tau0 (as if no cell were an
// obstacle), E01 and dist_to_target, each indexed by cell; tau0 / dt may be null.  Functions of (shape, start, target,
// parameters) only -- a batch of maps that share them shares the tables.
static void host_table_rows(int C, int start, int target, const mpp_maaco_params *p, int r_lo, int r_hi, double *tau0,
                            double *E01, double *dt) {
    const int sr = start / C, sc = start % C, tr = target / C, tc = target % C;
    double dsT = hdist(sr, sc, tr, tc);
    if (dsT < 1e-9) dsT = 1e-9;  // MAACO.py:43-45
    for (int r = r_lo; r < r_hi; ++r)
        for (int c = 0; c < C; ++c) {
            const size_t i = (size_t)r * C + c;
            const double diT = hdist(r, c, tr, tc);
            const double dsi = hdist(sr, sc, r, c);
            if (dt) dt[i] = diT;
            if (tau0) {
                const double den = dsi + diT;                // MAACO.py:58-84
                double factor;
                if (den < 1e-9) factor = (dsi < 1e-6 || diT < 1e-6) ? 1.0 : 0.1;
                else factor = dsT / den;
                const double v = factor * p->C0_initial_pheromone;
                tau0[i] = v < 1e-9 ? 1e-9 : v;
            }
            double h;                                        // MAACO.py:197-210
            if (dsT < 1e-9) h = p->wh_min;
            else h = p->wh_max - (p->wh_max - p->wh_min) * std::exp(-p->k_h_adaptive * diT / dsT);
            const double g = 1.0 - h;
            const double base = g * dsi + h * diT;
            double d0 = base + p->a_turn_coef * 0.0, d1 = base + p->a_turn_coef * 1.0;
            d0 = d0 > 1e-9 ? d0 : 1e-9;
            d1 = d1 > 1e-9 ? d1 : 1e-9;
            E01[2 * i] = std::pow(1.0 / d0, p->beta);        // turn flag 0
            E01[2 * i + 1] = std::pow(1.0 / d1, p->beta);    // turn flag 1
        }
}

// run work(lo, hi) over [0, n_items) on up to nt threads (nt <= 1: on the caller's thread)
template <class F>
static void host_parallel(long long n_items, unsigned nt, F work) {
    if (nt > n_items) nt = (unsigned)n_items;
    if (nt < 2) {
        work(0ll, n_items);
        return;
    }
    std::vector<std::thread> th;
    const long long per = (n_items + nt - 1) / nt;
    for (unsigned t = 0; t < nt; ++t) {
        const long long lo = (long long)t * per, hi = lo + per > n_items ? n_items : lo + per;
        if (lo < hi) th.emplace_back(work, lo, hi);
    }
    for (auto &t : th) t.join();
}

// the default thread count of the host table builds: at most 16, one thread below 65536 cells
static unsigned host_threads(size_t cells) {
    unsigned nt = std::thread::hardware_concurrency();
    if (nt > 16) nt = 16;
    return cells < 65536 ? 1u : nt;
}

static void host_tables(int R, int C, int start, int target, const mpp_maaco_params *p, double *tau0, double *E01,
                        double *dt) {
    host_parallel(R, host_threads((size_t)R * C), [&](long long lo, long long hi) {
        host_table_rows(C, start, target, p, (int)lo, (int)hi, tau0, E01, dt);
    });
}

extern "C" int mpp_maaco_e01_host(int rows, int cols, int n, const int32_t *start, const int32_t *target,
                                  const mpp_maaco_params *p, double *out, int threads) {
    MPP_REQUIRE(rows > 0 && cols > 0, "mpp_maaco_e01_host: bad shape %d x %d", rows, cols);
    MPP_REQUIRE(n >= 0, "mpp_maaco_e01_host: n = %d < 0", n);
    MPP_REQUIRE(threads >= 0, "mpp_maaco_e01_host: threads = %d < 0", threads);
    if (n == 0) return MPP_OK;
    MPP_REQUIRE(start && target && p && out, "mpp_maaco_e01_host: null argument");
    const long long cells = (long long)rows * cols;
    for (int k = 0; k < n; ++k)
        MPP_REQUIRE(start[k] >= 0 && start[k] < cells && target[k] >= 0 && target[k] < cells,
                    "mpp_maaco_e01_host: pair %d (start %d, target %d) is outside the %d x %d map", k, (int)start[k],
                    (int)target[k], rows, cols);
    // one work item = one row of one map: a batch spreads over its maps, a single map over its rows
    const unsigned nt = threads ? (unsigned)threads : host_threads((size_t)cells * n);
    try {
        host_parallel((long long)n * rows, nt, [&](long long lo, long long hi) {
            for (long long w = lo; w < hi;) {
                const int k = (int)(w / rows), r0 = (int)(w % rows);
                const int r1 = (int)std::min<long long>(rows, r0 + (hi - w));
                host_table_rows(cols, start[k], target[k], p, r0, r1, nullptr, out + (size_t)k * 2 * cells, nullptr);
                w += r1 - r0;
            }
        });
    } catch (const std::exception &e) {
        mpp_set_error("mpp_maaco_e01_host: %s", e.what());
        return MPP_ENOMEM;
    }
    return MPP_OK;
}

// tau0 of every map of the batch = the shared free-cell table with the map's obstacles at 1e-9 (MAACO.py:62-63)
__global__ void mpp_maaco_tau0_kernel(const double *__restrict__ tau0_free, const uint32_t *__restrict__ occ, int occ_words,
                                      int pitch, int R, int C, double *__restrict__ tau, long long tau_stride) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * C) return;
    occ += (size_t)blockIdx.y * occ_words;
    const int r = i / C, pb = i % C + 1;
    const bool obst = (occ[(r + 1) * pitch + (pb >> 5)] >> (pb & 31)) & 1u;
    tau[(size_t)blockIdx.y * tau_stride + i] = obst ? 1e-9 : tau0_free[i];
}

extern "C" int mpp_maaco_tables(const mpp_map_batch *maps, const mpp_maaco_params *p, double *tau0_dev, long long tau_stride,
                                double *E01_dev, double *dist_t_dev, void *stream) {
    MPP_REQUIRE(maps && p && tau0_dev && E01_dev, "mpp_maaco_tables: null argument");
    const int R = maps->rows, C = maps->cols;
    const size_t n = (size_t)R * C;
    MPP_REQUIRE(tau_stride >= (long long)n, "mpp_maaco_tables: tau_stride < rows*cols");
    const MppMapMeta &M0 = maps->meta_host[0];
    MPP_REQUIRE(M0.start >= 0 && M0.target >= 0, "mpp_maaco_tables: map has no start/target");
    for (int k = 1; k < maps->n_maps; ++k)
        MPP_REQUIRE(maps->meta_host[k].start == M0.start && maps->meta_host[k].target == M0.target,
                    "mpp_maaco_tables: the maps of a batch must share start and target (map %d differs); group them", k);
    std::vector<double> buf(4 * n);
    double *tau0 = buf.data(), *E01 = tau0 + n, *dt = E01 + 2 * n;
    host_tables(R, C, M0.start, M0.target, p, tau0, E01, dt);
    cudaStream_t s = (cudaStream_t)stream;
    MPP_CUDA(cudaSetDevice(maps->device));
    double *tau0_free = nullptr;
    MPP_CUDA(cudaMalloc(&tau0_free, n * 8));
    MPP_CUDA(cudaMemcpyAsync(tau0_free, tau0, n * 8, cudaMemcpyHostToDevice, s));
    MPP_CUDA(cudaMemcpyAsync(E01_dev, E01, 2 * n * 8, cudaMemcpyHostToDevice, s));
    if (dist_t_dev) MPP_CUDA(cudaMemcpyAsync(dist_t_dev, dt, n * 8, cudaMemcpyHostToDevice, s));
    mpp_maaco_tau0_kernel<<<dim3(((int)n + 255) / 256, maps->n_maps), 256, 0, s>>>(
        tau0_free, maps->occ_dev, maps->occ_words, maps->pitch_words, R, C, tau0_dev, tau_stride);
    MPP_CUDA(cudaGetLastError());
    MPP_CUDA(cudaStreamSynchronize(s));  // buf / tau0_free are released on return
    MPP_CUDA(cudaFree(tau0_free));
    return MPP_OK;
}

// tau0 of every map from its OWN start / target (MAACO.py:58-84, dsT floored as :43-45), obstacles at 1e-9 (:62-63):
// host_table_rows' expression with the same integer dr^2 + dc^2, correctly rounded sqrt and division and no FMA
// (-fmad=false), so each value is bit for bit what the host writes.
// MP (per-map parameters): C0 is params[k].C0_initial_pheromone instead of the launch's scalar.
template <bool MP>
__device__ __forceinline__ void tau0_maps_body(const MppMapMeta *__restrict__ meta, const uint32_t *__restrict__ occ,
                                               int occ_words, int pitch, int R, int C, double C0,
                                               const mpp_maaco_params *__restrict__ params, double *__restrict__ tau,
                                               long long tau_stride) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * C) return;
    const int k = blockIdx.y;
    if constexpr (MP) C0 = params[k].C0_initial_pheromone;
    occ += (size_t)k * occ_words;
    const int r = i / C, c = i % C, pb = c + 1;
    const int start = meta[k].start, target = meta[k].target;
    const int sr = start / C, sc = start % C, tr = target / C, tc = target % C;
    auto dist = [](int r0, int c0, int r1, int c1) {
        const long long dr = r0 - r1, dc = c0 - c1;
        return sqrt((double)(dr * dr + dc * dc));
    };
    double dsT = dist(sr, sc, tr, tc);
    if (dsT < 1e-9) dsT = 1e-9;
    const double diT = dist(r, c, tr, tc), dsi = dist(sr, sc, r, c);
    const double den = dsi + diT;
    double factor;
    if (den < 1e-9) factor = (dsi < 1e-6 || diT < 1e-6) ? 1.0 : 0.1;
    else factor = dsT / den;
    const double v = factor * C0;
    const bool obst = (occ[(r + 1) * pitch + (pb >> 5)] >> (pb & 31)) & 1u;
    tau[(size_t)k * tau_stride + i] = obst || v < 1e-9 ? 1e-9 : v;
}
__global__ void mpp_maaco_tau0_maps_kernel(const MppMapMeta *__restrict__ meta, const uint32_t *__restrict__ occ,
                                           int occ_words, int pitch, int R, int C, double C0, double *__restrict__ tau,
                                           long long tau_stride) {
    tau0_maps_body<false>(meta, occ, occ_words, pitch, R, C, C0, nullptr, tau, tau_stride);
}
__global__ void mpp_maaco_tau0_maps_p_kernel(const MppMapMeta *__restrict__ meta, const uint32_t *__restrict__ occ,
                                             int occ_words, int pitch, int R, int C,
                                             const mpp_maaco_params *__restrict__ params, double *__restrict__ tau,
                                             long long tau_stride) {
    tau0_maps_body<true>(meta, occ, occ_words, pitch, R, C, 0.0, params, tau, tau_stride);
}

// one of p (the launch's scalars) / params_dev (per map) is given; `who` names the entry point in errors
static int tau0_maps_launch(const mpp_map_batch *maps, const mpp_maaco_params *p, const mpp_maaco_params *params_dev,
                            double *tau0_dev, long long tau_stride, void *stream, const char *who) {
    MPP_REQUIRE(maps && (p || params_dev) && tau0_dev, "%s: null argument", who);
    const int R = maps->rows, C = maps->cols;
    const long long n = (long long)R * C;
    MPP_REQUIRE(tau_stride >= n, "%s: tau_stride < rows*cols", who);
    for (int k = 0; k < maps->n_maps; ++k)
        MPP_REQUIRE(maps->meta_host[k].start >= 0 && maps->meta_host[k].target >= 0, "%s: map %d has no start/target", who, k);
    if (maps->n_maps == 0) return MPP_OK;
    MPP_CUDA(cudaSetDevice(maps->device));
    const dim3 grid((unsigned)((n + 255) / 256), maps->n_maps);
    if (params_dev)
        mpp_maaco_tau0_maps_p_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
            maps->meta_dev, maps->occ_dev, maps->occ_words, maps->pitch_words, R, C, params_dev, tau0_dev, tau_stride);
    else
        mpp_maaco_tau0_maps_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
            maps->meta_dev, maps->occ_dev, maps->occ_words, maps->pitch_words, R, C, p->C0_initial_pheromone, tau0_dev,
            tau_stride);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

extern "C" int mpp_maaco_tau0_maps(const mpp_map_batch *maps, const mpp_maaco_params *p, double *tau0_dev,
                                   long long tau_stride, void *stream) {
    return tau0_maps_launch(maps, p, nullptr, tau0_dev, tau_stride, stream, "mpp_maaco_tau0_maps");
}

extern "C" int mpp_maaco_tau0_maps_p(const mpp_map_batch *maps, const mpp_maaco_params *params_dev, double *tau0_dev,
                                     long long tau_stride, void *stream) {
    MPP_REQUIRE(params_dev, "mpp_maaco_tau0_maps_p: null params_dev");
    return tau0_maps_launch(maps, nullptr, params_dev, tau0_dev, tau_stride, stream, "mpp_maaco_tau0_maps_p");
}

// E01 of every map from its OWN start / target (MAACO.py:197-210, dsT floored as :43-45): host_table_rows' expression
// in its order -- integer dr^2 + dc^2, correctly rounded sqrt and division, no FMA (-fmad=false) -- with mpp_exp /
// mpp_pow for libm's exp / pow, so each value is bit for bit what mpp_maaco_e01_host writes.
template <bool MP>
__device__ __forceinline__ void e01_maps_body(const MppMapMeta *__restrict__ meta, int R, int C, double beta,
                                              double wh_max, double wh_min, double k_h, double a_turn,
                                              const mpp_maaco_params *__restrict__ params, double *__restrict__ E01,
                                              long long E01_stride) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * C) return;
    const int k = blockIdx.y;
    if constexpr (MP) {
        const mpp_maaco_params &P = params[k];
        beta = P.beta; wh_max = P.wh_max; wh_min = P.wh_min; k_h = P.k_h_adaptive; a_turn = P.a_turn_coef;
    }
    const int r = i / C, c = i % C;
    const int start = meta[k].start, target = meta[k].target;
    const int sr = start / C, sc = start % C, tr = target / C, tc = target % C;
    auto dist = [](int r0, int c0, int r1, int c1) {
        const long long dr = r0 - r1, dc = c0 - c1;
        return sqrt((double)(dr * dr + dc * dc));
    };
    double dsT = dist(sr, sc, tr, tc);
    if (dsT < 1e-9) dsT = 1e-9;
    const double diT = dist(r, c, tr, tc), dsi = dist(sr, sc, r, c);
    const double h = wh_max - (wh_max - wh_min) * mpp_exp(-k_h * diT / dsT);
    const double g = 1.0 - h;
    const double base = g * dsi + h * diT;
    double d0 = base + a_turn * 0.0, d1 = base + a_turn * 1.0;
    d0 = d0 > 1e-9 ? d0 : 1e-9;
    d1 = d1 > 1e-9 ? d1 : 1e-9;
    *(double2 *)(E01 + (size_t)k * E01_stride + 2 * (size_t)i) = make_double2(mpp_pow(1.0 / d0, beta), mpp_pow(1.0 / d1, beta));
}
__global__ void mpp_maaco_e01_maps_kernel(const MppMapMeta *__restrict__ meta, int R, int C, double beta, double wh_max,
                                          double wh_min, double k_h, double a_turn, double *__restrict__ E01,
                                          long long E01_stride) {
    e01_maps_body<false>(meta, R, C, beta, wh_max, wh_min, k_h, a_turn, nullptr, E01, E01_stride);
}
// MP: beta, a_turn_coef, wh_max, wh_min, k_h_adaptive of params[k]
__global__ void mpp_maaco_e01_maps_p_kernel(const MppMapMeta *__restrict__ meta, int R, int C,
                                            const mpp_maaco_params *__restrict__ params, double *__restrict__ E01,
                                            long long E01_stride) {
    e01_maps_body<true>(meta, R, C, 0.0, 0.0, 0.0, 0.0, 0.0, params, E01, E01_stride);
}

static int e01_maps_launch(const mpp_map_batch *maps, const mpp_maaco_params *p, const mpp_maaco_params *params_dev,
                           double *E01_dev, long long E01_stride, void *stream, const char *who) {
    MPP_REQUIRE(maps && (p || params_dev) && E01_dev, "%s: null argument", who);
    const int R = maps->rows, C = maps->cols;
    const long long n = (long long)R * C;
    MPP_REQUIRE(E01_stride >= 2 * n && E01_stride % 2 == 0, "%s: E01_stride %lld is odd or < 2*rows*cols", who, E01_stride);
    MPP_REQUIRE(((uintptr_t)E01_dev & 15) == 0, "%s: E01_dev is not 16-byte aligned", who);
    for (int k = 0; k < maps->n_maps; ++k)
        MPP_REQUIRE(maps->meta_host[k].start >= 0 && maps->meta_host[k].target >= 0, "%s: map %d has no start/target", who, k);
    if (maps->n_maps == 0) return MPP_OK;
    MPP_CUDA(cudaSetDevice(maps->device));
    const dim3 grid((unsigned)((n + 255) / 256), maps->n_maps);
    if (params_dev)
        mpp_maaco_e01_maps_p_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(maps->meta_dev, R, C, params_dev, E01_dev,
                                                                             E01_stride);
    else
        mpp_maaco_e01_maps_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
            maps->meta_dev, R, C, p->beta, p->wh_max, p->wh_min, p->k_h_adaptive, p->a_turn_coef, E01_dev, E01_stride);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

extern "C" int mpp_maaco_e01_maps(const mpp_map_batch *maps, const mpp_maaco_params *p, double *E01_dev,
                                  long long E01_stride, void *stream) {
    return e01_maps_launch(maps, p, nullptr, E01_dev, E01_stride, stream, "mpp_maaco_e01_maps");
}

extern "C" int mpp_maaco_e01_maps_p(const mpp_map_batch *maps, const mpp_maaco_params *params_dev, double *E01_dev,
                                    long long E01_stride, void *stream) {
    MPP_REQUIRE(params_dev, "mpp_maaco_e01_maps_p: null params_dev");
    return e01_maps_launch(maps, nullptr, params_dev, E01_dev, E01_stride, stream, "mpp_maaco_e01_maps_p");
}

__global__ void mpp_libm_exp_pow_kernel(int n, const double *__restrict__ e, const double *__restrict__ x,
                                        const double *__restrict__ y, double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[2 * (size_t)i] = mpp_exp(e[i]);
    out[2 * (size_t)i + 1] = mpp_pow(x[i], y[i]);
}

extern "C" int mpp_libm_exp_pow(int n, const double *e, const double *x, const double *y, double *out, int device,
                                void *stream) {
    MPP_REQUIRE(n >= 0, "mpp_libm_exp_pow: n = %d < 0", n);
    if (n == 0) return MPP_OK;
    MPP_REQUIRE(e && x && y && out, "mpp_libm_exp_pow: null argument");
    MPP_CUDA(cudaSetDevice(device));
    mpp_libm_exp_pow_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n, e, x, y, out);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

// ---------------------------------------------------------------------------------------------
// sizes
// ---------------------------------------------------------------------------------------------
// Ranking buffer layout (uint32 words): [margin | 9*R*C strategy-1 words | margin | pad to even] [9*R*C full entries
// (2 words)] [pad to 4] [R*C bundles of 4 words: word2 of the three cells P1's moves lead to, ready for one 16-byte load]
// [R*C x 8 bytes: for each of the eight moves the packed word2 of the cell it leads to (context = that move), what a
// tier-3 step needs to go on without a dependent load].  The margins let the tour kernel read the word of a neighbour
// cell without bounds checks.
struct RankLayout { size_t margin, fast_words, bundle_words, nb8_words, total_words; };
static RankLayout rank_layout(int R, int C) {
    RankLayout L;
    L.margin = (size_t)(C + 2) * 9;
    L.fast_words = ((size_t)9 * R * C + 2 * L.margin + 1) & ~(size_t)1;
    L.bundle_words = (L.fast_words + (size_t)18 * R * C + 3) & ~(size_t)3;
    L.nb8_words = L.bundle_words + (size_t)4 * R * C;
    L.total_words = L.nb8_words + (size_t)2 * R * C;
    return L;
}
static inline int tiles_r(int R) { return (R + 31) >> 5; }
static inline int tiles_c(int C) { return (C + 31) >> 5; }

extern "C" long long mpp_maaco_rank_words(int rows, int cols) { return (long long)rank_layout(rows, cols).total_words; }
extern "C" long long mpp_maaco_slab_words(int tile_rows, int cols, int n_ants) {
    return (long long)tile_rows * tiles_c(cols) * (long long)n_ants * 32;
}
extern "C" long long mpp_maaco_touched_words(int tile_rows, int cols, int n_ants) {
    return 2ll * tile_rows * tiles_c(cols) * ((n_ants + 31) / 32);
}

// ---------------------------------------------------------------------------------------------
// K2: tour construction, one thread per ant.  One ant step is a serial chain (position -> tabu bits -> candidate
// set -> selection -> position) and a colony pass lasts as long as its longest tour times the latency of that
// chain, so the chain stays inside ONE thread (no shuffles / votes / warp reductions on it) and touches only
// shared memory; a lone warp issues about one instruction per 5 cycles here, so what counts is the number of
// instructions on the chain and every exposed memory latency (profiles/r01_tour1_summary.md):
//   * tabu bits (:93-95) come from a 64x64-cell WINDOW of the ant's visited set in shared memory (rows of two
//     words; the ant stays at least U cells inside it).  A global store to a line evicts it from L1 (measured:
//     tools/ubench/l1_store.cu, 123 -> 432 cycles per dependent load), so re-reading a bitmap the ant itself
//     keeps writing costs an L2 round trip per step wherever it lives in global memory.  When the ant reaches
//     the window's edge the window slides by one 32-cell tile: the warp writes the two leaving tiles to the ant's
//     slabs (one coalesced 128-byte store each, skipped when the tile is empty) and reloads the entering ones if
//     the ant has been there before (`touched` bit); the four tiles still in the window are written at the end;
//   * strategy 1 (:165, almost every step): the strategy-1 word of (cell, previous move) from mpp_maaco_rank
//     -- static move mask + what greedy selection keeps of every subset of P1's three moves -- plus the
//     precomputed greedy flag / floor(u1*n) of the step index one shared-memory table row that yields the move
//     and all its deltas.  The words of the three possible next cells are prefetched one step ahead;
//   * every other step (no strategy-1 candidate, P1 without three moves, a cell whose attractiveness is not
//     tiny): all eight moves, strategies 2/3, the full ranking entry or the literal rules (tour_select_slow);
//   * the warp's lanes generate Philox blocks together: lane L makes the block of ant L%apw, step s+L/apw.
// `apw` lanes of each warp own an ant: fewer ants per warp = more warps to spread over the SMs.
// ---------------------------------------------------------------------------------------------
#define MPP_MAX_PEERS 16
extern "C" int mpp_maaco_max_peers(void) { return MPP_MAX_PEERS; }
struct TourArgs {
    const MppMapMeta *meta;      // [n_maps]
    const uint32_t *rank;        // [n_maps][rank_stride] ranking buffers (mpp_maaco_rank), layout: rank_layout()
    size_t rank_stride, rank_margin, rank_fast_words, rank_bundle_words, rank_nb8_words;
    int R, C;
    const double *tau, *E01;
    size_t tau_stride, E01_stride;
    uint32_t it;
    double q0, alpha;
    int n_ants, ant_offset;
    const uint64_t *seeds;       // [n_maps]
    uint32_t *slabs, *touched;   // this pass's buffers
    size_t slab_stride, touched_stride;
    uint8_t *moves;
    int max_cells;
    mpp_ant_result *result;
    size_t result_stride;        // results of one map (>= ant_offset + n_ants)
    unsigned long long *steps;
    const int32_t *latch;        // non-zero = a sharded colony's exchange overflowed: every kernel is a no-op until the host rewinds
};
// sharded colony over peer memory (mpp_maaco_tours_p2p, the kernel's P2P instantiation): every slab the kernel writes also
// goes, over NVLink, straight into the receive buffers of the rank that updates that tile row, and every result into every
// rank's table (the pointers travel in the kernel parameters: a slide must not wait for a global load to learn where to store)
struct TourPeers {
    uint32_t *peer_slabs[MPP_MAX_PEERS];       // slabs_recv of each rank: [its tile rows x TC][n_total][32]
    uint32_t *peer_touched[MPP_MAX_PEERS];     // touched_recv of each rank (both parities)
    mpp_ant_result *peer_result[MPP_MAX_PEERS];   // result table of each rank [n_total]
    int n_peers, rows_per_rank;      // tile rows per rank
    int n_total;                     // ants of the whole colony
};

#define MPP_SQRT2 1.4142135623730951  // sqrt(2.0) correctly rounded == math.sqrt(2)
#ifndef MPP_TOUR1_THREADS
#define MPP_TOUR1_THREADS 128
#endif

__device__ __noinline__ double pow_slow(double x, double y) { return pow(x, y); }

// literal selection rules MAACO.py:228-262 for one ant; cand = candidate move mask (move order :98).
__device__ __noinline__ int tour_select_slow(uint32_t cand, int cr, int cc, int C, bool have_prev, int prev_m,
                                             const double *__restrict__ tau, const double *__restrict__ E01,
                                             double alpha, double q0, double u0, double u1) {
    int mv[8], n = 0;
    double attr[8];
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        if (!((cand >> m) & 1u)) continue;
        const int dr = (int)((0xA940u >> (2 * m)) & 3u) - 1, dc = (int)((0x9224u >> (2 * m)) & 3u) - 1;
        const int j = (cr + dr) * C + (cc + dc);
        const bool turn = have_prev && (m != prev_m);                 // :184-195
        const double tv = tau[j];
        const double ta = (alpha == 1.0) ? tv : pow_slow(tv, alpha);
        attr[n] = ta * E01[2 * (size_t)j + (turn ? 1 : 0)];           // :238
        mv[n] = m;
        ++n;
    }
    int k;
    if (u0 <= q0) {                                                   // greedy :241-250
        double mx = -1.0;
        int best[8], nb = 0;
        for (int i = 0; i < n; ++i) {
            if (attr[i] > mx) { mx = attr[i]; nb = 0; best[nb++] = i; }
            else if (fabs(attr[i] - mx) < 1e-9) best[nb++] = i;
        }
        int q = (int)(u1 * (double)nb);
        q = q < nb ? q : nb - 1;
        k = best[q];
    } else {
        double S = 0.0;                                               // :252 plain left-to-right
        for (int i = 0; i < n; ++i) S += attr[i];
        bool uniform = S < 1e-9;                                      // :253-254
        double pr[8];
        double ps = 0.0;
        if (!uniform) {
            for (int i = 0; i < n; ++i) { pr[i] = attr[i] / S; ps += pr[i]; }   // :255
            if (fabs(ps - 1.0) > 1e-6) {                              // :257-258
                const double ps0 = ps;
                ps = 0.0;
                for (int i = 0; i < n; ++i) { pr[i] = pr[i] / ps0; ps += pr[i]; }
            }
            if (!(fabs(ps - 1.0) <= 1.4901161193847656e-08)) uniform = true;    // choice() ValueError -> :262
        }
        if (uniform) {
            k = (int)(u1 * (double)n);
        } else {
            // RandomState.choice: cdf = cumsum(p); cdf /= cdf[-1]; searchsorted(u, side='right')
            double cdf[8], acc = 0.0;
            for (int i = 0; i < n; ++i) { acc += pr[i]; cdf[i] = acc; }
            k = 0;
            for (int i = 0; i < n; ++i)
                if (cdf[i] / acc <= u1) ++k;
        }
        k = k < n ? k : n - 1;
    }
    return mv[k];
}

// One 32x32-cell tile of ant `a`'s visited set, lane = tile row.  Warp-level: all 32 lanes call these together.
struct TourSlabs {
    uint32_t *slabs, *touched;   // of this map
    size_t n_ants;
    int NW, TR, TC;
    const TourPeers *peers;                              // null unless the colony is sharded over peer memory
    int rows_per_rank, ant_offset, NW_total;
    size_t n_total, peer_touched_off;                    // this pass's parity inside a rank's touched_recv
};
__device__ __forceinline__ uint32_t tour_tile_load(const TourSlabs &V, int a, int trow, int tcx, int lane) {
    if (trow < 0 || trow >= V.TR || tcx < 0 || tcx >= V.TC) return 0u;
    const int tile = trow * V.TC + tcx;
    // the bit was set (if at all) by lane 0 of this warp: lane 0 reads it back, program order on one address
    uint32_t tw = 0u;
    if (lane == 0) tw = __ldcg(V.touched + (size_t)tile * V.NW + (a >> 5));
    tw = __shfl_sync(0xffffffffu, tw, 0);
    if (!((tw >> (a & 31)) & 1u)) return 0u;
    return __ldcg(V.slabs + ((size_t)tile * V.n_ants + a) * 32 + lane);      // row `lane` was stored by this lane
}
__device__ __forceinline__ void tour_tile_store(const TourSlabs &V, int a, int trow, int tcx, int lane, uint32_t v) {
    if (trow < 0 || trow >= V.TR || tcx < 0 || tcx >= V.TC) return;
    if (!__any_sync(0xffffffffu, v != 0u)) return;                           // nothing visited in this tile
    const int tile = trow * V.TC + tcx;
    V.slabs[((size_t)tile * V.n_ants + a) * 32 + lane] = v;                  // one 128-byte line
    if (lane == 0) atomicOr(V.touched + (size_t)tile * V.NW + (a >> 5), 1u << (a & 31));
    if (V.peers) {
        // the same line for the rank that updates this tile row (possibly this one): a peer store + a peer reduction,
        // neither waited for; a tile that is stored again later in the tour (the ant came back) carries a superset
        const int g = trow / V.rows_per_rank, tl = (trow - g * V.rows_per_rank) * V.TC + tcx;
        const size_t ga = (size_t)V.ant_offset + a;
        V.peers->peer_slabs[g][((size_t)tl * V.n_total + ga) * 32 + lane] = v;
        if (lane == 0) atomicOr(V.peers->peer_touched[g] + V.peer_touched_off + (size_t)tl * V.NW_total + (ga >> 5), 1u << (ga & 31));
    }
}

// a load the compiler may not sink to its use (it would turn "select among three loaded entries" into "one load
// from the selected address" and put the L2 latency back on the ant's serial chain)
__device__ __forceinline__ uint32_t ldg32_pinned(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// shared-memory loads by 32-bit shared address (kept in registers; the generic form re-derives the window base)
__device__ __forceinline__ uint2 lds_u2(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

// shared-memory tables of the tour kernel (per block)
struct Tour1Move {          // one per move (order MAACO.py:98)
    int dcur;               // flat cell delta  dr*C + dc
    int dprow;              // byte delta of the window row pointer  dr*8
    int dc;                 // column delta
    int dphi;               // change of the start->target potential  dr*sgn(tr-sr) + dc*sgn(tc-sc)
};
#define T1_KTH_OFF 0                        // uint8  kth[256*8]   : index of the k-th set bit
#define T1_SPREAD_OFF 2048                  // uint2  spread[256]  : byte m = 0xFF if bit m set
#define T1_MOVE_OFF 4096                    // Tour1Move move[8]
#define T1_DLEN_OFF (4096 + 128)            // double dlen[8]      : 1.0 or sqrt(2) (:293)
#define T1_FAST_OFF (4096 + 256)            // uint4 fast[4]       : member of P1 -> {dcur, dprow, dc, move | dphi << 8}
#define T1_FLEN_OFF (4096 + 256 + 64)       // double flen[4]      : step length of that member
#define T1_FLD_OFF (4096 + 256 + 96)        // uint32 fld[8]      : fields [24:4] of word2 for each order of P1's members (nb8 bytes)
#define T1_RNG_OFF (4096 + 256 + 128)       // per warp: double2 u[32] (512 B) + uint32 pack[32] + uint32 pack2[32]
#define T1_RNG_BYTES 768
#define T1_WIN_OFF (T1_RNG_OFF + (MPP_TOUR1_THREADS / 32) * T1_RNG_BYTES)

// Strategy-1 word, second form ("word2": what the tour's fast tiers work on; made from the ranking word by
// tour_word2).  P1's three moves are "members" 0..2 (move order).  [0] 1 = the ranking does not apply here (some
// attractiveness >= 1e-10); [3:1] A = members that are statically possible from this cell; [24:4] for every non-empty
// candidate subset c (field c-1) what greedy selection keeps of it; [27:25] G = what it keeps of A.
__device__ __forceinline__ uint32_t tour_word2(uint32_t w, int sm0, int sm1, int sm2) {
    const uint32_t sv = w >> 24;
    const uint32_t A3 = ((sv >> sm0) & 1u) | (((sv >> sm1) & 1u) << 1) | (((sv >> sm2) & 1u) << 2);
    const uint32_t G = A3 ? ((w >> (3u * A3)) & 7u) : 0u;
    return ((w & 7u) ? 1u : 0u) | (A3 << 1) | (((w >> 3) & 0x1FFFFFu) << 4) | (G << 25);
}
// The same word in one byte (the nb8 table): [0] ranking n/a, [3:1] A, [6:4] how the ranking orders P1's three members
// (bit 4: member 0 before 1, bit 5: 0 before 2, bit 6: 1 before 2); the fields follow from the order (tour_fields).
__host__ __device__ __forceinline__ uint32_t tour_fields(uint32_t order) {
    const uint32_t b01 = order & 1u, b02 = (order >> 1) & 1u, b12 = (order >> 2) & 1u;
    const uint32_t p0 = (1u - b01) + (1u - b02), p1 = b01 + (1u - b12), p2 = b02 + b12;   // members ranked before it
    uint32_t f = 0u;
    for (uint32_t c = 1; c < 8; ++c) {
        uint32_t bp = 8u, bi = 0u;
        if ((c & 1u) && p0 < bp) { bp = p0; bi = 0u; }
        if ((c & 2u) && p1 < bp) { bp = p1; bi = 1u; }
        if ((c & 4u) && p2 < bp) { bp = p2; bi = 2u; }
        f |= (c & ~((1u << bi) - 1u)) << (3u * (c - 1u));
    }
    return f;
}
// the prefetch of the three possible next cells' word2 (one 16-byte line of the bundle table), pinned where it is issued
__device__ __forceinline__ uint4 ldg128_pinned(const uint4 *p) {
    uint4 v;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint2 ldg64_pinned(const uint2 *p) {
    uint2 v;
    asm volatile("ld.global.nc.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ldg32_nc_pinned(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

#ifndef MPP_TOUR1_MINB
#define MPP_TOUR1_MINB 4
#endif
struct TourNoPeers {};
// per-map colony parameters (the kernel's MP instantiation, mpp_maaco_pass_maps): alpha of params[map] and q0 of the
// pass's row of the q0 table instead of TourArgs' scalars; they travel in the third parameter, which P2P never combines with
struct TourMapParams {
    const mpp_maaco_params *params;  // [n_maps]
    const double *q0;                // [n_maps] this pass's q0 of every map
    const int32_t *sizes;            // [n_maps][2] {num_ants, num_iterations} of every map, or null (mpp_maaco_pass_maps_sized)
};
// Map m's colony under a sizes array (the MP instantiations): sizes[m].num_ants clamped to [0, cap], where cap is the
// launch's n_ants (the buffers' ant capacity), so no value can index past them.  Map m takes part in pass k only
// while k <= sizes[m].num_iterations.
__device__ __forceinline__ int sized_ants(const int32_t *sizes, int map, int cap) {
    const int n = sizes[2 * map];
    return n < 0 ? 0 : (n < cap ? n : cap);
}
__device__ __forceinline__ bool sized_past(const int32_t *sizes, int map, int iteration) {
    return iteration > sizes[2 * map + 1];
}
template <bool P2P, bool MP>
using TourExtra = typename std::conditional<P2P, TourPeers, typename std::conditional<MP, TourMapParams, TourNoPeers>::type>::type;
template <bool P2P, bool MP>
__global__ void __launch_bounds__(MPP_TOUR1_THREADS, MPP_TOUR1_MINB)
mpp_maaco_tour1_kernel(const TourArgs A, const int apw, const TourExtra<P2P, MP> PA) {
    static_assert(!(P2P && MP), "a sharded colony has one parameter set");
    extern __shared__ __align__(16) uint8_t t1_smem[];
    if (A.latch && *A.latch) return;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int R = A.R, C = A.C, TC = (C + 31) >> 5;
    const int map = blockIdx.y;
    // MP with sizes: a map past its pass count constructs nothing (the whole CTA: grid.y = map), and only the map's own
    // colony of n_live ants runs, writes slabs and results and counts steps.  (Read as `MP ? n_live : A.n_ants`, like
    // k_q0 below.)
    int n_live = A.n_ants;
    if constexpr (MP) {
        if (PA.sizes) {
            if (sized_past(PA.sizes, map, (int)A.it)) return;
            n_live = sized_ants(PA.sizes, map, A.n_ants);
        }
    }
    // MP: the same for the whole CTA (grid.y = map), loaded once and held in registers through the step loop.  (Read as
    // `MP ? k_q0 : A.q0`: the other instantiations keep reading TourArgs' scalars exactly as before.)
    double k_q0 = 0.0, k_alpha = 0.0;
    if constexpr (MP) {
        k_q0 = __shfl_sync(0xffffffffu, PA.q0[map], 0);
        k_alpha = __shfl_sync(0xffffffffu, PA.params[map].alpha, 0);
    }
    const MppMapMeta &MM = A.meta[map];
    const MppS1 s1 = MM.s1;
    const int target = MM.target;
    const int tr = target / C, tc = target % C;
    {   // ---- tables ----
        const int sgr = (tr > MM.start / C) - (tr < MM.start / C), sgc = (tc > MM.start % C) - (tc < MM.start % C);
        uint8_t *const kth = t1_smem + T1_KTH_OFF;
        uint2 *const spread = (uint2 *)(t1_smem + T1_SPREAD_OFF);
        for (int p = threadIdx.x; p < 256; p += MPP_TOUR1_THREADS) {
            int idx = 0;
            uint32_t lo = 0, hi = 0;
            for (int b = 0; b < 8; ++b)
                if ((p >> b) & 1) {
                    kth[p * 8 + idx++] = (uint8_t)b;
                    if (b < 4) lo |= 0xFFu << (8 * b); else hi |= 0xFFu << (8 * (b - 4));
                }
            for (; idx < 8; ++idx) kth[p * 8 + idx] = 0;
            spread[p] = make_uint2(lo, hi);
        }
        if (threadIdx.x < 8) {
            const int m = threadIdx.x;
            const int dr = (int)((0xA940u >> (2 * m)) & 3u) - 1, dc = (int)((0x9224u >> (2 * m)) & 3u) - 1;
            Tour1Move mv;
            mv.dcur = dr * C + dc; mv.dprow = dr * 8; mv.dc = dc; mv.dphi = dr * sgr + dc * sgc;
            ((Tour1Move *)(t1_smem + T1_MOVE_OFF))[m] = mv;
            ((double *)(t1_smem + T1_DLEN_OFF))[m] = (dr != 0 && dc != 0) ? MPP_SQRT2 : 1.0;
        }
        if (threadIdx.x < 4) {                                     // member of P1's three moves -> everything the move implies
            const int k = threadIdx.x < 3 ? threadIdx.x : 2;
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            double dl = 1.0;
            if (s1.fast_ok) {
                const int mm = s1.sm[k];
                const int dr = (int)((0xA940u >> (2 * mm)) & 3u) - 1, dc = (int)((0x9224u >> (2 * mm)) & 3u) - 1;
                v = make_uint4((uint32_t)(dr * C + dc), (uint32_t)(dr * 8), (uint32_t)dc,
                               (uint32_t)mm | ((uint32_t)(dr * sgr + dc * sgc) << 8));      // dphi = 1 or 2 for P1 moves
                dl = (dr != 0 && dc != 0) ? MPP_SQRT2 : 1.0;
            }
            ((uint4 *)(t1_smem + T1_FAST_OFF))[threadIdx.x] = v;
            ((double *)(t1_smem + T1_FLEN_OFF))[threadIdx.x] = dl;
        }
        if (threadIdx.x >= 32 && threadIdx.x < 40) ((uint32_t *)(t1_smem + T1_FLD_OFF))[threadIdx.x - 32] = tour_fields(threadIdx.x - 32);
    }
    double2 *const rngu = (double2 *)(t1_smem + T1_RNG_OFF + wib * T1_RNG_BYTES);
    uint32_t *const rngp = (uint32_t *)(t1_smem + T1_RNG_OFF + wib * T1_RNG_BYTES + 512);
    uint32_t *const rngq = (uint32_t *)(t1_smem + T1_RNG_OFF + wib * T1_RNG_BYTES + 640);
    uint2 *const win_w = (uint2 *)(t1_smem + T1_WIN_OFF) + (size_t)wib * apw * 64;   // the warp's windows: 64 rows x uint2 each
    for (int i = lane; i < apw * 64; i += 32) win_w[i] = make_uint2(0u, 0u);          // a tour starts with nothing visited
    __syncthreads();
    const int warp = (blockIdx.x * MPP_TOUR1_THREADS + threadIdx.x) >> 5;
    const int a0 = warp * apw;                                     // first ant of this warp
    if (a0 >= (MP ? n_live : A.n_ants)) return;                    // whole warp
    const int a = a0 + lane;
    bool active = lane < apw && a < (MP ? n_live : A.n_ants);
    int cur = MM.start;
    auto orient_mask = [](int dR, int dC) -> uint32_t {           // MAACO.py:146-157
        uint32_t k = 0xffu;
        if (dC > 0) k &= ~0x29u;
        if (dC < 0) k &= ~0x94u;
        if (dR > 0) k &= ~0x07u;
        if (dR < 0) k &= ~0xE0u;
        return k;
    };
    const uint32_t P1 = s1.P1;                                     // the same for every ant of a map
    const bool fast_ok = s1.fast_ok;                               // P1 has 3 moves unless start and target share a row or column
    // (kept in registers: re-reading them inside the step costs a memory round trip each time)
#define T1_KEEP(x) x = __shfl_sync(0xffffffffu, x, 0)   /* a value ptxas cannot re-derive from its source */
    int k_sm0 = s1.sm[0], k_sm1 = s1.sm[1], k_sm2 = s1.sm[2], k_dpr0 = s1.dpr[0], k_dpr1 = s1.dpr[1], k_dpr2 = s1.dpr[2];
    int k_dc0 = s1.dc[0], k_dc1 = s1.dc[1], k_dc2 = s1.dc[2];
    T1_KEEP(k_sm0); T1_KEEP(k_sm1); T1_KEEP(k_sm2); T1_KEEP(k_dpr0); T1_KEEP(k_dpr1); T1_KEEP(k_dpr2);
    T1_KEEP(k_dc0); T1_KEEP(k_dc1); T1_KEEP(k_dc2);
    TourSlabs V;
    V.slabs = A.slabs + (size_t)map * A.slab_stride;
    V.touched = A.touched + (size_t)map * A.touched_stride;
    V.n_ants = (size_t)A.n_ants; V.NW = (A.n_ants + 31) >> 5; V.TR = (R + 31) >> 5; V.TC = TC;
    V.peers = nullptr;
    V.rows_per_rank = 1; V.ant_offset = A.ant_offset; V.n_total = 0; V.NW_total = 0; V.peer_touched_off = 0;
    if constexpr (P2P) {
        V.peers = &PA;
        V.rows_per_rank = PA.rows_per_rank; V.n_total = (size_t)PA.n_total;
        V.NW_total = (PA.n_total + 31) >> 5;
        V.peer_touched_off = (size_t)(A.it & 1u) * (size_t)PA.rows_per_rank * TC * (size_t)V.NW_total;
    }
    uint8_t *mvp = A.moves + ((size_t)map * A.n_ants + (active ? a : a0)) * A.max_cells;   // next move-code slot
    const double *const tau_m = A.tau + (size_t)map * A.tau_stride;
    const double *const E01_m = A.E01 + (size_t)map * A.E01_stride;
    const uint32_t *__restrict__ rank_fast = A.rank + (size_t)map * A.rank_stride + A.rank_margin;
    const uint2 *const rank_slow = (const uint2 *)(A.rank + (size_t)map * A.rank_stride + A.rank_fast_words);
    const uint4 *bundle = (const uint4 *)(A.rank + (size_t)map * A.rank_stride + A.rank_bundle_words);
    const uint2 *const nb8 = (const uint2 *)(A.rank + (size_t)map * A.rank_stride + A.rank_nb8_words);
    {
        unsigned long long bf = (unsigned long long)bundle;
        bf = __shfl_sync(0xffffffffu, bf, 0);
        bundle = (const uint4 *)bf;
    }
    int k_target = target, k_max_cells = A.max_cells, k_max_path = 2 * R * C + 1;   // step cap 2*R*C (MAACO.py:283); R*C < 2^30
    T1_KEEP(k_target); T1_KEEP(k_max_cells); T1_KEEP(k_max_path);
    const uint64_t seed = A.seeds[map];
    const uint32_t key0 = (uint32_t)seed, key1 = (uint32_t)(seed >> 32);
    int n_path = 1, prev_m = -1, turns = -1;                       // (the first move is counted as a "turn": hence -1)
    double len = 0.0;
    bool failed = false;
    // The start -> target potential phi = r*sgn(tr-sr) + c*sgn(tc-sc) grows with every move of P1, so while the ant
    // stands on the largest phi it has ever reached (gap == 0) none of P1's target cells can have been visited:
    // the tabu test (:93-95) of a strategy-1 step is then `gap == 0` instead of three window loads.
    int gap = 0;                                                   // max phi reached - phi of the current cell
#ifdef MPP_TOUR_STATS
    int st_t1 = 0, st_t2 = 0, st_t3 = 0, st_slides = 0;
    const long long st_c0 = clock64();
    long long st_c1 = st_c0;
#endif
    // window = tile rows {wr, wr+1} x tile cols {wc, wc+1} (64 x 64 cells); row lrow of it is the uint2 at prow,
    // bit lcol of that 64-bit row is the cell; the ant stays in [1, 62] x [1, 62]
    int wr, wc, lrow, lcol;
    {
        const int cr = cur / C, cc = cur % C;
        wr = (cr >> 5) - (((cr & 31) < 16) ? 1 : 0);
        wc = (cc >> 5) - (((cc & 31) < 16) ? 1 : 0);
        lrow = cr - (wr << 5);
        lcol = cc - (wc << 5);
    }
    uint32_t prow_s = (uint32_t)__cvta_generic_to_shared(win_w + (size_t)(lane < apw ? lane : 0) * 64 + lrow);   // the ant's window row
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(t1_smem);
    const uint32_t rngp_s = (uint32_t)__cvta_generic_to_shared(rngp) + 4u * (uint32_t)lane;
    const uint32_t rngq_s = (uint32_t)__cvta_generic_to_shared(rngq) + 4u * (uint32_t)lane;
    uint32_t sbase_k = sbase;                                    // (opaque copy: otherwise re-derived from %cluster_ctaid every use)
    sbase_k = __shfl_sync(0xffffffffu, sbase_k, 0);
    uint32_t fw2 = 1u;                                            // word2 of (cell, previous move); 1 = "no fast tier here"
    uint4 bq = make_uint4(1u, 1u, 1u, 1u);                        // word2 of the three strategy-1 neighbours, prefetched
    if (active) {
        asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(prow_s + 4u * ((uint32_t)lcol >> 5)), "r"(1u << (lcol & 31)) : "memory");
        if (cur == target) active = false;
        if (fast_ok) {
            fw2 = tour_word2(rank_fast[(size_t)cur * 9], k_sm0, k_sm1, k_sm2);   // context 0: no previous move
            bq = ldg128_pinned(bundle + cur);
        }
    }
    __syncwarp();
    const uint32_t gmask = (uint32_t)(32 / apw) - 1u;              // a cooperative Philox pass covers 32/apw steps
    // U steps per pass of the warp-level bookkeeping below (liveness vote, Philox refill, window slides): an ant may
    // then be U cells from where the checks saw it, so the window keeps a margin of U cells instead of one
    const int U = (apw <= 16) ? 2 : 1;                             // a refill covers 32 / apw steps: must be a multiple of U
    const unsigned edge_lo = (unsigned)U, edge_span = 63u - 2u * (unsigned)U;
    const uint32_t slot_bytes = 4u * (uint32_t)apw;
    for (uint32_t step = 0;; step += (uint32_t)U) {
        const uint32_t need0 = __ballot_sync(0xffffffffu, active && ((unsigned)lrow - edge_lo > edge_span || (unsigned)lcol - edge_lo > edge_span));
        if (!__any_sync(0xffffffffu, active)) break;
        if ((step & gmask) == 0 || need0) {
            if ((step & gmask) == 0) {
                // uniforms: draws 2s (q-test) and 2s+1 (selection) of stream (seed, TOUR, it, ant) = Philox block s;
                // lane L makes the block of ant L % apw for step + L / apw.  Besides u0/u1 (for the literal rules) the
                // pass leaves what the ranked tiers need: the greedy flag u0 <= q0 (:240), floor(u1 * n) for every
                // pool size n = 1..8 (random.choice on n items: `pack`), and for every subset of P1's three members
                // the member random.choice picks from it (`pack2`, two bits per subset; bit 16 = greedy flag).
                const int la = lane & (apw - 1);
                const mpp_u4 rb = mpp_philox(step + (uint32_t)(lane / apw), (uint32_t)(A.ant_offset + a0 + la), A.it,
                                             MPP_CLS_MAACO_TOUR, key0, key1);
                const double u0 = mpp_u53(rb.x, rb.y), u1 = mpp_u53(rb.z, rb.w);
                const bool greedy = u0 <= (MP ? k_q0 : A.q0);
                uint32_t pack = greedy ? (1u << 24) : 0u;
#pragma unroll
                for (int n = 2; n <= 8; ++n) {
                    int k = (int)(u1 * (double)n);
                    k = k < n ? k : n - 1;
                    pack |= (uint32_t)k << (3 * (n - 1));
                }
                const uint32_t k2 = (pack >> 3) & 7u, k3 = (pack >> 6) & 7u;     // floor(u1*2), floor(u1*3)
                // subsets 1,2,4: the only member; 3 = {0,1}, 5 = {0,2}, 6 = {1,2}: k2-th; 7: k3-th
                uint32_t pack2 = (greedy ? (1u << 16) : 0u) | (0u << 2) | (1u << 4) | (2u << 8);
                pack2 |= (k2 ? 1u : 0u) << 6;
                pack2 |= (k2 ? 2u : 0u) << 10;
                pack2 |= (k2 ? 2u : 1u) << 12;
                pack2 |= k3 << 14;
                __syncwarp();
                rngu[lane] = make_double2(u0, u1);
                rngp[lane] = pack;
                rngq[lane] = pack2;
                __syncwarp();
            }
            // ---- slide the windows whose ant reached their edge (at most every 31 steps per ant) ----
            uint32_t need = need0;
            while (need) {
                const int src = __ffs(need) - 1;
                const int s_lrow = __shfl_sync(0xffffffffu, lrow, src), s_lcol = __shfl_sync(0xffffffffu, lcol, src);
                const int s_wr = __shfl_sync(0xffffffffu, wr, src), s_wc = __shfl_sync(0xffffffffu, wc, src);
                const int a_s = a0 + src;
                uint2 *const w_s = win_w + src * 64;
                int d_wr = 0, d_wc = 0;
                if ((unsigned)s_lrow - edge_lo > edge_span) {      // vertical: one tile row leaves, one enters
                    const bool up = s_lrow < U;
                    d_wr = up ? -1 : 1;
                    const int t_out = up ? s_wr + 1 : s_wr, t_in = up ? s_wr - 1 : s_wr + 2;
                    const uint2 keep = w_s[up ? lane : lane + 32], out = w_s[up ? lane + 32 : lane];
                    tour_tile_store(V, a_s, t_out, s_wc, lane, out.x);
                    tour_tile_store(V, a_s, t_out, s_wc + 1, lane, out.y);
                    uint2 nw;
                    nw.x = tour_tile_load(V, a_s, t_in, s_wc, lane);
                    nw.y = tour_tile_load(V, a_s, t_in, s_wc + 1, lane);
                    w_s[up ? lane + 32 : lane] = keep;
                    w_s[up ? lane : lane + 32] = nw;
                } else {                                           // horizontal: the two words of each row shift
                    const bool left = s_lcol < U;
                    d_wc = left ? -1 : 1;
                    const int t_out = left ? s_wc + 1 : s_wc, t_in = left ? s_wc - 1 : s_wc + 2;
                    const uint2 o0 = w_s[lane], o1 = w_s[lane + 32];
                    tour_tile_store(V, a_s, s_wr, t_out, lane, left ? o0.y : o0.x);
                    tour_tile_store(V, a_s, s_wr + 1, t_out, lane, left ? o1.y : o1.x);
                    const uint32_t x0 = tour_tile_load(V, a_s, s_wr, t_in, lane);
                    const uint32_t x1 = tour_tile_load(V, a_s, s_wr + 1, t_in, lane);
                    w_s[lane] = left ? make_uint2(x0, o0.x) : make_uint2(o0.y, x0);
                    w_s[lane + 32] = left ? make_uint2(x1, o1.x) : make_uint2(o1.y, x1);
                }
#ifdef MPP_TOUR_STATS
                if (lane == src) ++st_slides;
#endif
                if (lane == src) {
                    wr += d_wr; wc += d_wc;
                    lrow -= d_wr << 5; lcol -= d_wc << 5;
                    prow_s -= (uint32_t)(d_wr * 256);
                }
                __syncwarp();
                // a diagonal step can leave through a corner: this ant may still need the other direction
                const bool again = (lane == src) && ((unsigned)lrow - edge_lo > edge_span || (unsigned)lcol - edge_lo > edge_span);
                need = (need & (need - 1)) | __ballot_sync(0xffffffffu, again);
            }
        }
        uint32_t slot = (step & gmask) * slot_bytes;               // byte offset of this step's slot in the warp's rng arrays
        for (int su = 0; su < U; ++su, slot += slot_bytes)
        if (active) {
            int m = -1, dcur = 0, dpr = 0, dcc = 0, dphi = 0;         // the move taken this step and what it implies
            double dl = 0.0;
            // ---- tiers 1 and 2: strategy 1 (:165) on the three moves of P1, from the prefetched word2 ----
            if (!(fw2 & 1u)) {
                const uint32_t p2 = lds_u32(rngq_s + slot);
                const uint32_t A3 = (fw2 >> 1) & 7u;                              // static candidates among P1's members
                uint32_t pool;
#ifdef MPP_TOUR_STATS
                if (gap == 0) ++st_t1; else ++st_t2;
#endif
                if (gap == 0) {
                    // tier 1: nothing ahead can be tabu.  greedy (:241-250) keeps G of A; roulette (:251-254) all of A
                    pool = (p2 & 0x10000u) ? ((fw2 >> 25) & 7u) : A3;
                } else {
                    // tier 2: tabu bits (:93-95) of the three target cells from the window
                    const uint2 ra = lds_u2(prow_s + k_dpr0), rb = lds_u2(prow_s + k_dpr1), rc = lds_u2(prow_s + k_dpr2);
                    const int c0 = lcol + k_dc0, c1 = lcol + k_dc1, c2 = lcol + k_dc2;           // 0..63
                    const uint32_t v0 = ((c0 & 32) ? ra.y : ra.x) >> (c0 & 31);
                    const uint32_t v1 = ((c1 & 32) ? rb.y : rb.x) >> (c1 & 31);
                    const uint32_t v2 = ((c2 & 32) ? rc.y : rc.x) >> (c2 & 31);
                    const uint32_t c3 = A3 & ~((v0 & 1u) | ((v1 & 1u) << 1) | ((v2 & 1u) << 2));
                    pool = (p2 & 0x10000u) ? ((fw2 >> (1u + 3u * c3)) & 7u) : c3;   // (c3 == 0: field -1 -> bits of A, masked below)
                    if (c3 == 0u) pool = 0u;
                }
                if (pool != 0u) {
                    // random.choice (:250 / :254): the member chosen from `pool`, and everything the move implies
                    const uint32_t mem = (p2 >> (2u * pool)) & 3u;
                    const uint4 fv = lds_u4(sbase_k + T1_FAST_OFF + 16u * mem);
                    dl = lds_f64(sbase_k + T1_FLEN_OFF + 8u * mem);
                    dcur = (int)fv.x; dpr = (int)fv.y; dcc = (int)fv.z;
                    m = (int)(fv.w & 0xFFu);
                    dphi = (int)(fv.w >> 8);
                    // word2 of the cell moved to: one of the three prefetched (bitwise select, opaque to the compiler:
                    // as a ternary the default operand is copied early and that copy waits for the prefetch too soon)
                    const uint32_t m1 = 0u - (mem & 1u), m2 = 0u - (mem >> 1);
                    uint32_t t;
                    asm("lop3.b32 %0, %1, %2, %3, 0xD8;" : "=r"(t) : "r"(bq.x), "r"(bq.y), "r"(m1));
                    asm("lop3.b32 %0, %1, %2, %3, 0xD8;" : "=r"(fw2) : "r"(t), "r"(bq.z), "r"(m2));
                }
            }
#ifdef MPP_TOUR_STATS
            if (m < 0) { ++st_t3; if (!(fw2 & 1u)) { if (gap == 0) --st_t1; else --st_t2; } }
#endif
            if (m < 0) {
                // ---- tier 3: all eight moves, strategies 1-3, full ranking entry or the literal rules ----
                const uint32_t ctx = (n_path >= 2) ? (uint32_t)(prev_m + 1) : 0u;
                // everything the step may need from the ranking tables is requested at once (one L2 round trip instead of
                // up to three in a row): the ranking word and the full entry of (cell, previous move), and the packed word2
                // of all eight neighbours for the step after this one
                const uint32_t fw = ldg32_nc_pinned(rank_fast + (size_t)cur * 9 + ctx);
                const uint2 rws = ldg64_pinned(rank_slow + (size_t)cur * 9 + ctx);
                uint2 nb = make_uint2(0u, 0u);
                if (fast_ok) nb = ldg64_pinned(nb8 + cur);
                const uint32_t pack = lds_u32(rngp_s + slot);
                const uint2 q0r = lds_u2(prow_s - 8u), q1r = lds_u2(prow_s), q2r = lds_u2(prow_s + 8u);
                const int rot = lcol - 1;                             // 0..61
                const bool sw = rot & 32;
                const uint32_t t3 = __funnelshift_r(sw ? q0r.y : q0r.x, q0r.y, rot) & 7u;
                const uint32_t m3 = __funnelshift_r(sw ? q1r.y : q1r.x, q1r.y, rot) & 5u;
                const uint32_t b3 = __funnelshift_r(sw ? q2r.y : q2r.x, q2r.y, rot) & 7u;
                const uint32_t vis = t3 | ((m3 & 1u) << 3) | ((m3 & 4u) << 2) | (b3 << 5);
                const uint32_t valid = (fw >> 24) & ~vis;             // static mask (:93-120) minus tabu (:93-95)
                uint32_t cand = valid & P1;                           // strategy 1 :165
                if (cand == 0u) {
                    cand = valid & orient_mask(tr - cur / C, tc - cur % C);   // strategy 2 :169
                    if (!cand) cand = valid;                          // strategy 3 :172-180
                }
                if (cand == 0u) {                                     // :287-288
                    failed = true;
                    active = false;
                } else {
                    if ((cand & (cand - 1u)) == 0u) {
                        m = __ffs(cand) - 1;                          // one candidate: every rule picks it
                    } else if ((fw & 7u) != 0u) {                     // some attractiveness >= 1e-10: literal rules
                        const double2 uu = rngu[(slot >> 2) + lane];
                        m = tour_select_slow(cand, cur / C, cur % C, C, n_path >= 2, prev_m, tau_m, E01_m, MP ? k_alpha : A.alpha,
                                         MP ? k_q0 : A.q0, uu.x, uu.y);
                    } else {
                        uint32_t pool = cand;                         // roulette over tiny values: uniform (:253-254)
                        if (pack & (1u << 24)) {
                            // greedy: first arg-max = best-ranked candidate (full entry: permute the candidate flags
                            // into rank order, take the first) and every later candidate
                            const uint2 sp = lds_u2(sbase_k + T1_SPREAD_OFF + 8u * cand);
                            const uint32_t f0 = __byte_perm(sp.x, sp.y, rws.x & 0xFFFFu), f1 = __byte_perm(sp.x, sp.y, rws.x >> 16);
                            const uint32_t ff = f0 ? f0 : f1;
                            const int pos4 = ((__ffs(ff) - 1) >> 1) + (f0 ? 0 : 16);
                            const uint32_t best = (rws.x >> pos4) & 7u;
                            pool = cand & ~((1u << best) - 1u);
                        }
                        const int n = __popc(pool);
                        const int k = (pack >> (3 * n - 3)) & 7u;
                        m = (int)lds_u8(sbase_k + T1_KTH_OFF + pool * 8u + (uint32_t)k);
                    }
                    const uint4 mvv = lds_u4(sbase_k + T1_MOVE_OFF + 16u * (uint32_t)m);
                    dcur = (int)mvv.x; dpr = (int)mvv.y; dcc = (int)mvv.z; dphi = (int)mvv.w;
                    dl = lds_f64(sbase_k + T1_DLEN_OFF + 8u * (uint32_t)m);
                    if (fast_ok) {
                        const uint32_t by = (((m & 4) ? nb.y : nb.x) >> (8 * (m & 3))) & 0xFFu;   // packed word2 of the cell moved to
                        const uint32_t fl = lds_u32(sbase_k + T1_FLD_OFF + 4u * (by >> 4));
                        const uint32_t A3n = (by >> 1) & 7u;
                        const uint32_t Gn = A3n ? ((fl >> (3u * (A3n - 1u))) & 7u) : 0u;
                        fw2 = (by & 1u) | (A3n << 1) | (fl << 4) | (Gn << 25);
                    }
                }
            }
            if (active) {
                // ---- advance :293-297 ----
                cur += dcur;
                if (fast_ok) bq = ldg128_pinned(bundle + cur);        // the three possible next cells' word2: a step ahead
                gap -= dphi;
                gap = gap > 0 ? gap : 0;
                prow_s += (uint32_t)dpr;
                lrow += dpr >> 3;
                lcol += dcc;
                asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(prow_s + 4u * ((uint32_t)lcol >> 5)), "r"(1u << (lcol & 31)) : "memory");
                if (n_path <= k_max_cells) *mvp = (uint8_t)m;         // move code of step n_path-1
                ++mvp;
                len += dl;                                            // :293 (1.0 or sqrt(2), plain += in path order)
                if (m != prev_m) ++turns;                             // :264-276 counted on the fly
                prev_m = m;
                ++n_path;
                if (cur == k_target || n_path >= k_max_path) active = false;
#ifdef MPP_TOUR_STATS
                st_c1 = clock64();
#endif
            }
        }
    }
    // ---- the windows still hold the marks of their four tiles: write them to the ants' slabs ----
    for (int src = 0; src < apw && a0 + src < (MP ? n_live : A.n_ants); ++src) {
        const int s_wr = __shfl_sync(0xffffffffu, wr, src), s_wc = __shfl_sync(0xffffffffu, wc, src);
        const uint2 o0 = win_w[src * 64 + lane], o1 = win_w[src * 64 + lane + 32];
        tour_tile_store(V, a0 + src, s_wr, s_wc, lane, o0.x);
        tour_tile_store(V, a0 + src, s_wr, s_wc + 1, lane, o0.y);
        tour_tile_store(V, a0 + src, s_wr + 1, s_wc, lane, o1.x);
        tour_tile_store(V, a0 + src, s_wr + 1, s_wc + 1, lane, o1.y);
    }
    if (lane < apw && a < (MP ? n_live : A.n_ants)) {
        const bool ok = !failed && cur == target;
        mpp_ant_result res;
        res.length = ok ? len : __longlong_as_double(0x7ff0000000000000ll);
        res.n_cells = ok ? n_path : 0;
        res.turns = ok ? (turns > 0 ? turns : 0) : -1;
        A.result[(size_t)map * A.result_stride + A.ant_offset + a] = res;
        if constexpr (P2P)
            for (int g = 0; g < PA.n_peers; ++g) PA.peer_result[g][A.ant_offset + a] = res;
        if (A.steps) atomicAdd(A.steps, (unsigned long long)(n_path - 1));
#ifdef MPP_TOUR_STATS
        int *st = (int *)(A.moves + ((size_t)map * A.n_ants + a + 1) * A.max_cells - 32);
        st[0] = st_t1; st[1] = st_t2; st[2] = st_t3; st[3] = st_slides; st[4] = (int)(st_c1 - st_c0); st[5] = n_path - 1;
        st[6] = ok ? 1 : 0;
#endif
    }
}

static int colony_check(const mpp_map_batch *maps, const mpp_colony *c, const char *who) {
    MPP_REQUIRE(maps && c, "%s: null argument", who);
    MPP_REQUIRE(c->tau && c->E01 && c->rank && c->slabs && c->touched && c->moves && c->result && c->deposit && c->okbits &&
                    c->state && c->best_cells && c->seeds, "%s: null colony buffer", who);
    MPP_REQUIRE(c->max_cells > 0 && c->tau_stride >= (long long)maps->rows * maps->cols, "%s: bad max_cells / tau_stride", who);
    for (int k = 0; k < maps->n_maps; ++k)
        MPP_REQUIRE(maps->meta_host[k].start >= 0 && maps->meta_host[k].target >= 0, "%s: map %d has no start/target", who, k);
    return MPP_OK;
}

static int tours_launch(const mpp_map_batch *maps, const mpp_colony *c, int iteration, double q0, double alpha,
                        int n_ants, int ant_offset, int n_ants_total, int ants_per_warp,
                        uint32_t *const *peer_slabs, uint32_t *const *peer_touched, mpp_ant_result *const *peer_result,
                        int n_peers, int rows_per_rank, void *stream, const TourMapParams *mp = nullptr) {
    int rc = colony_check(maps, c, "mpp_maaco_tours");
    if (rc) return rc;
    MPP_REQUIRE(n_ants > 0 && ant_offset >= 0 && ant_offset + n_ants <= n_ants_total, "mpp_maaco_tours: bad ant range");
    MPP_CUDA(cudaSetDevice(maps->device));
    const RankLayout L = rank_layout(maps->rows, maps->cols);
    const int TR = tiles_r(maps->rows);
    TourArgs A;
    A.meta = maps->meta_dev;
    A.rank = c->rank; A.rank_stride = L.total_words; A.rank_margin = L.margin; A.rank_fast_words = L.fast_words;
    A.rank_bundle_words = L.bundle_words; A.rank_nb8_words = L.nb8_words;
    A.R = maps->rows; A.C = maps->cols;
    A.tau = c->tau; A.tau_stride = (size_t)c->tau_stride; A.E01 = c->E01; A.E01_stride = (size_t)c->E01_stride;
    A.it = (uint32_t)iteration; A.q0 = q0; A.alpha = alpha;
    A.n_ants = n_ants; A.ant_offset = ant_offset;
    A.seeds = c->seeds;
    const size_t tw = (size_t)mpp_maaco_touched_words(TR, maps->cols, n_ants) / 2;   // one parity, one map
    A.slabs = c->slabs; A.slab_stride = (size_t)mpp_maaco_slab_words(TR, maps->cols, n_ants);
    A.touched = c->touched + (size_t)(iteration & 1) * tw * maps->n_maps; A.touched_stride = tw;
    A.moves = c->moves; A.max_cells = c->max_cells;
    A.result = c->result; A.result_stride = (size_t)n_ants_total;
    A.steps = c->steps; A.latch = c->latch;
    TourPeers PA;
    for (int g = 0; g < MPP_MAX_PEERS; ++g) {
        PA.peer_slabs[g] = g < n_peers ? peer_slabs[g] : nullptr;
        PA.peer_touched[g] = g < n_peers ? peer_touched[g] : nullptr;
        PA.peer_result[g] = g < n_peers ? peer_result[g] : nullptr;
    }
    PA.n_peers = n_peers; PA.rows_per_rank = rows_per_rank; PA.n_total = n_ants_total;
    // ants per warp: enough warps for every SM sub-partition first, full warps only for big colonies
    int apw = 16;                                                  // measured (tools/batch_time.py): 16 beats 32 even at 131 k ants
    const char *e = getenv("MPP_TOUR_APW");
    if (e) apw = atoi(e);
    else if (ants_per_warp) apw = ants_per_warp;
    else {
        const long long total = (long long)n_ants * maps->n_maps;
        while (apw > 2 && (total + apw - 1) / apw < 12ll * maps->sm_count) apw >>= 1;   // measured: 2 ants/warp at 4096 ants
    }
    MPP_REQUIRE(apw == 1 || apw == 2 || apw == 4 || apw == 8 || apw == 16 || apw == 32,
                "ants per warp (MPP_TOUR_APW / ants_per_warp) must be a power of two <= 32");
    const int warps = (n_ants + apw - 1) / apw, wpb = MPP_TOUR1_THREADS / 32;
    const size_t smem = T1_WIN_OFF + (size_t)wpb * apw * 512;   // tables + per-warp RNG + 512-byte windows
    {   // raise the kernel's dynamic shared-memory limit only when it grows (the call is slow; devices tracked apart)
        static size_t smem_set[64] = {0};
        const int dv = maps->device & 63;
        if (smem > smem_set[dv]) {
            MPP_CUDA(cudaFuncSetAttribute(mpp_maaco_tour1_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            MPP_CUDA(cudaFuncSetAttribute(mpp_maaco_tour1_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            MPP_CUDA(cudaFuncSetAttribute(mpp_maaco_tour1_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            smem_set[dv] = smem;
        }
    }
    const dim3 grid((warps + wpb - 1) / wpb, maps->n_maps);
    if (mp) mpp_maaco_tour1_kernel<false, true><<<grid, MPP_TOUR1_THREADS, smem, (cudaStream_t)stream>>>(A, apw, *mp);
    else if (n_peers > 0) mpp_maaco_tour1_kernel<true, false><<<grid, MPP_TOUR1_THREADS, smem, (cudaStream_t)stream>>>(A, apw, PA);
    else mpp_maaco_tour1_kernel<false, false><<<grid, MPP_TOUR1_THREADS, smem, (cudaStream_t)stream>>>(A, apw, TourNoPeers());
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

extern "C" int mpp_maaco_tours(const mpp_map_batch *maps, const mpp_colony *c, int iteration, double q0, double alpha,
                               int n_ants, int ant_offset, int n_ants_total, int ants_per_warp, void *stream) {
    return tours_launch(maps, c, iteration, q0, alpha, n_ants, ant_offset, n_ants_total, ants_per_warp, nullptr, nullptr,
                        nullptr, 0, 1, stream);
}

extern "C" int mpp_maaco_tours_p2p(const mpp_map_batch *maps, const mpp_colony *c, int iteration, double q0, double alpha,
                                   int n_ants, int ant_offset, int n_ants_total, int ants_per_warp,
                                   uint32_t *const *slabs_peers, uint32_t *const *touched_peers,
                                   mpp_ant_result *const *result_peers, int n_peers, int tile_rows_per_rank, void *stream) {
    MPP_REQUIRE(maps && maps->n_maps == 1, "mpp_maaco_tours_p2p: a sharded colony is one map");
    MPP_REQUIRE(slabs_peers && touched_peers && result_peers && n_peers > 0 && n_peers <= MPP_MAX_PEERS && tile_rows_per_rank > 0 &&
                    (long long)n_peers * tile_rows_per_rank >= tiles_r(maps->rows), "mpp_maaco_tours_p2p: bad peer arguments");
    return tours_launch(maps, c, iteration, q0, alpha, n_ants, ant_offset, n_ants_total, ants_per_warp, slabs_peers,
                        touched_peers, result_peers, n_peers, tile_rows_per_rank, stream);
}

// ---------------------------------------------------------------------------------------------
// K2a: per (cell, turn context) ranking of the 8 moves by attractiveness tau**alpha * eta'**beta (MAACO.py:238).
// With beta = 7 the values are ~1e-8..1e-20, so the selection rules (:241-262) only depend on their ORDER
// (|attr_i - max| < 1e-9 and sum < 1e-9 always hold); the tour kernel then needs one word per step
// instead of 16 fp64 loads.  Context 0 = no previous move (turn flag 0 for every candidate, :185-186),
// context p+1 = previous move p (turn flag = (m != p)).  Entry = two words.  Word 1: [31:24] static move mask,
// [23:0] rank position of each move (0 = largest attractiveness, ties -> lower move index, exactly the order the
// sequential scan sees), or 0xFFFFFF when some attractiveness is >= 1e-10 (the tour kernel then applies the full
// rule).  Word 0: the inverse permutation, nibble p = move at rank position p (a PRMT selector).
//
// Strategy-1 word (one per (cell, context)): [31:24] static move mask; field c (3 bits at 3c, c = 1..7 = a subset of
// P1's three moves in move order) = what greedy selection (:241-250) keeps of candidate set c, as a subset again;
// field 0 = 0 when the ranking applies (all attractiveness < 1e-10), 7 when it does not; fields 1..7 are only
// filled when P1 has exactly three moves.
// ---------------------------------------------------------------------------------------------
// MP (per-map parameters): alpha of params[map] instead of the launch's scalar; with sizes, a map past its pass count
// is skipped (its tours return before they read the ranking)
template <bool MP>
__device__ __forceinline__ void rank_body(const uint8_t *__restrict__ svalid_all, const double *__restrict__ tau_all,
                                          size_t tau_stride, const double *__restrict__ E01_all, size_t E01_stride,
                                          double alpha, const mpp_maaco_params *__restrict__ params,
                                          const int32_t *__restrict__ sizes, int iteration, int R, int C,
                                          const MppMapMeta *__restrict__ meta, uint32_t *__restrict__ rank_all,
                                          size_t rank_stride, size_t rank_margin, size_t rank_fast_words,
                                          size_t rank_bundle_words, size_t rank_nb8_words,
                                          const int32_t *__restrict__ latch, const unsigned tid) {
    // one thread per cell: the eight neighbours' tau / eta' are read once and serve all nine contexts
    const int cell = blockIdx.x * 128 + tid;
    if (cell >= R * C) return;
    if (latch && *latch) return;
    const int map = blockIdx.y;
    if constexpr (MP) {
        if (sizes && sized_past(sizes, map, iteration)) return;
        alpha = params[map].alpha;
    }
    const uint8_t *svalid = svalid_all + (size_t)map * R * C;
    const double *tau = tau_all + (size_t)map * tau_stride;
    const double *E01 = E01_all + (size_t)map * E01_stride;
    uint32_t *rank_fast = rank_all + (size_t)map * rank_stride + rank_margin;
    uint2 *rank_slow = (uint2 *)(rank_all + (size_t)map * rank_stride + rank_fast_words);
    uint32_t *bundle = rank_all + (size_t)map * rank_stride + rank_bundle_words;
    uint8_t *nb8 = (uint8_t *)(rank_all + (size_t)map * rank_stride + rank_nb8_words);
    const uint32_t P1 = meta[map].s1.P1;
    const uint32_t sv = svalid[cell];
    double a0[8], a1[8];                                          // attractiveness without / with the turn factor (:238)
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        a0[m] = a1[m] = -1.0;
        if ((sv >> m) & 1u) {
            const int j = cell + ((int)((0xA940u >> (2 * m)) & 3u) - 1) * C + ((int)((0x9224u >> (2 * m)) & 3u) - 1);
            const double tv = tau[j];
            const double ta = (alpha == 1.0) ? tv : pow_slow(tv, alpha);
            const double2 e = *(const double2 *)(E01 + 2 * (size_t)j);
            a0[m] = ta * e.x;
            a1[m] = ta * e.y;
        }
    }
    const bool p1_three = __popc(P1) == 3;
    const int s0 = __ffs(P1) - 1, s1 = __ffs(P1 & (P1 - 1)) - 1, s2 = 31 - __clz(P1);
    for (int ctx = 0; ctx < 9; ++ctx) {
        double a[8];
#pragma unroll
        for (int m = 0; m < 8; ++m) a[m] = (ctx > 0 && m != ctx - 1) ? a1[m] : a0[m];   // turn flag :184-195
        // "small" is decided per context on the values that context uses (as the tour's full rule would see them)
        double cmx = 0.0;
#pragma unroll
        for (int m = 0; m < 8; ++m) cmx = fmax(cmx, a[m]);
        uint32_t word = 0xFFFFFFu, perm = 0u, fast = 7u, order = 0u;
        if (cmx < 1e-10) {
            word = 0u;
#pragma unroll
            for (int m = 0; m < 8; ++m) {
                int pos = 0;
#pragma unroll
                for (int q = 0; q < 8; ++q) pos += (a[q] > a[m]) || (a[q] == a[m] && q < m);
                word |= (uint32_t)pos << (3 * m);
                perm |= (uint32_t)m << (4 * pos);
            }
            fast = 0u;                                            // field 0: the ranking applies
            if (p1_three) {
                const uint32_t p0 = (word >> (3 * s0)) & 7u, p1 = (word >> (3 * s1)) & 7u, p2 = (word >> (3 * s2)) & 7u;
                order = (p0 < p1 ? 1u : 0u) | (p0 < p2 ? 2u : 0u) | (p1 < p2 ? 4u : 0u);
#pragma unroll
                for (uint32_t c = 1; c < 8; ++c) {
                    // best-ranked member of subset c (rank positions are distinct)
                    uint32_t bp = 8u, bi = 0u;
                    if ((c & 1u) && p0 < bp) { bp = p0; bi = 0u; }
                    if ((c & 2u) && p1 < bp) { bp = p1; bi = 1u; }
                    if ((c & 4u) && p2 < bp) { bp = p2; bi = 2u; }
                    fast |= (c & ~((1u << bi) - 1u)) << (3u * c);     // the best one and every later member
                }
            }
        }
        const size_t t = (size_t)cell * 9 + ctx;
        rank_fast[t] = fast | (sv << 24);
        rank_slow[t] = make_uint2(perm, word | (sv << 24));
        if (p1_three && ctx > 0) {
            // the cell this one is entered from by move ctx-1: its nb8 entry gets the packed word, and when the move is
            // P1's member k its bundle gets the word itself
            const int mv = ctx - 1;
            const int pr = cell / C - ((int)((0xA940u >> (2 * mv)) & 3u) - 1), pc = cell % C - ((int)((0x9224u >> (2 * mv)) & 3u) - 1);
            if (pr >= 0 && pr < R && pc >= 0 && pc < C) {
                const uint32_t A3 = ((sv >> s0) & 1u) | (((sv >> s1) & 1u) << 1) | (((sv >> s2) & 1u) << 2);
                nb8[((size_t)pr * C + pc) * 8 + mv] = (uint8_t)((fast & 7u ? 1u : 0u) | (A3 << 1) | (order << 4));
                const int k = (ctx == s0 + 1) ? 0 : ((ctx == s1 + 1) ? 1 : ((ctx == s2 + 1) ? 2 : -1));
                if (k >= 0) bundle[((size_t)pr * C + pc) * 4 + k] = tour_word2(fast | (sv << 24), s0, s1, s2);
            }
        }
    }
}
__global__ void __launch_bounds__(128) mpp_maaco_rank_kernel(const uint8_t *__restrict__ svalid_all,
                                                             const double *__restrict__ tau_all, size_t tau_stride,
                                                             const double *__restrict__ E01_all, size_t E01_stride,
                                                             double alpha, int R, int C,
                                                             const MppMapMeta *__restrict__ meta, uint32_t *__restrict__ rank_all,
                                                             size_t rank_stride, size_t rank_margin, size_t rank_fast_words,
                                                             size_t rank_bundle_words, size_t rank_nb8_words,
                                                             const int32_t *__restrict__ latch) {
    rank_body<false>(svalid_all, tau_all, tau_stride, E01_all, E01_stride, alpha, nullptr, nullptr, 0, R, C, meta, rank_all,
                     rank_stride, rank_margin, rank_fast_words, rank_bundle_words, rank_nb8_words, latch, threadIdx.x);
}
__global__ void __launch_bounds__(128) mpp_maaco_rank_p_kernel(const uint8_t *__restrict__ svalid_all,
                                                               const double *__restrict__ tau_all, size_t tau_stride,
                                                               const double *__restrict__ E01_all, size_t E01_stride,
                                                               const mpp_maaco_params *__restrict__ params,
                                                               const int32_t *__restrict__ sizes, int iteration, int R, int C,
                                                               const MppMapMeta *__restrict__ meta,
                                                               uint32_t *__restrict__ rank_all, size_t rank_stride,
                                                               size_t rank_margin, size_t rank_fast_words,
                                                               size_t rank_bundle_words, size_t rank_nb8_words,
                                                               const int32_t *__restrict__ latch) {
    rank_body<true>(svalid_all, tau_all, tau_stride, E01_all, E01_stride, 0.0, params, sizes, iteration, R, C, meta, rank_all,
                    rank_stride, rank_margin, rank_fast_words, rank_bundle_words, rank_nb8_words, latch, threadIdx.x);
}

// params_dev != null: the per-map instantiation (alpha of each map's params; sizes_dev: maps past their pass count skip)
static int rank_launch(const mpp_map_batch *maps, const mpp_colony *c, double alpha, const mpp_maaco_params *params_dev,
                       void *stream, const int32_t *sizes_dev = nullptr, int iteration = 0) {
    int rc = colony_check(maps, c, "mpp_maaco_rank");
    if (rc) return rc;
    MPP_CUDA(cudaSetDevice(maps->device));
    const int total = maps->rows * maps->cols;
    const RankLayout L = rank_layout(maps->rows, maps->cols);
    const dim3 grid((total + 127) / 128, maps->n_maps);
    if (params_dev)
        mpp_maaco_rank_p_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(
            maps->svalid_dev, c->tau, (size_t)c->tau_stride, c->E01, (size_t)c->E01_stride, params_dev, sizes_dev, iteration,
            maps->rows, maps->cols, maps->meta_dev, c->rank, L.total_words, L.margin, L.fast_words, L.bundle_words,
            L.nb8_words, c->latch);
    else
        mpp_maaco_rank_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(
            maps->svalid_dev, c->tau, (size_t)c->tau_stride, c->E01, (size_t)c->E01_stride, alpha, maps->rows, maps->cols,
            maps->meta_dev, c->rank, L.total_words, L.margin, L.fast_words, L.bundle_words, L.nb8_words, c->latch);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

extern "C" int mpp_maaco_rank(const mpp_map_batch *maps, const mpp_colony *c, double alpha, void *stream) {
    return rank_launch(maps, c, alpha, nullptr, stream);
}

// ---------------------------------------------------------------------------------------------
// K4: iteration-best / overall-best (MAACO.py:343-358) + deposits (:307-308) + the "deposits at all" bitmap the
// pheromone update filters its ant lists with; one block per map
// ---------------------------------------------------------------------------------------------
#define MPP_BEST_THREADS 1024
__device__ __forceinline__ bool lt_len_idx(double la, int ia, double lb, int ib) {
    return la < lb || (la == lb && ia < ib);
}
__device__ __forceinline__ int move_delta(uint32_t m, int C) {
    return ((int)((0xA940u >> (2 * m)) & 3u) - 1) * C + ((int)((0x9224u >> (2 * m)) & 3u) - 1);
}

// MP (per-map parameters): Q of params[map] instead of the launch's scalar; with sizes, a map past its pass count keeps
// its state, best path and log, and the scans see only the map's own colony (ants [n_live, n) deposit nothing)
template <bool MP>
__device__ __forceinline__ void best_body(const mpp_ant_result *__restrict__ res_all, const uint8_t *__restrict__ moves_all,
                                          int max_cells, int moves_ant_offset, int moves_n_ants, int n, double Q,
                                          const mpp_maaco_params *__restrict__ params, const int32_t *__restrict__ sizes,
                                          int iteration, int C,
                                          const MppMapMeta *__restrict__ meta, mpp_maaco_state *state_all,
                                          int32_t *best_cells_all, double *deposit_all, uint32_t *okbits_all,
                                          double *log_all, int log_rows, const int32_t *__restrict__ latch) {
    __shared__ double s_len[32];
    __shared__ int s_idx[32];
    __shared__ int s_t[32];
    __shared__ double b_len;
    __shared__ int b_r, b_ant, b_turns, b_copy, s_base;
    if (latch && *latch) return;
    const int map = blockIdx.x;
    int n_live = n;
    if constexpr (MP) {
        if (sizes) {
            if (sized_past(sizes, map, iteration)) return;              // the whole CTA (one block per map)
            n_live = sized_ants(sizes, map, n);
        }
        Q = params[map].Q;
    }
    const mpp_ant_result *res = res_all + (size_t)map * n;
    double *deposit = deposit_all + (size_t)map * n;
    uint32_t *okbits = okbits_all + (size_t)map * ((n + 31) >> 5);
    mpp_maaco_state *state = state_all + map;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const double INF = __longlong_as_double(0x7ff0000000000000ll);
    // phase 1: global min length and its first index r (the last strict record of the scan)
    double ml = INF;
    int mi = 0x7fffffff;
    for (int i0 = 0; i0 < n; i0 += MPP_BEST_THREADS) {               // whole warps stay together for the ballot
        const int i = i0 + tid;
        bool dep = false;
        if (i < n_live) {
            const mpp_ant_result ri = res[i];
            const double l = ri.length;
            if (lt_len_idx(l, i, ml, mi)) { ml = l; mi = i; }
            // deposit amount MAACO.py:307-308 (0.0 == "does not deposit"; x + 0.0 is exact anyway)
            dep = (l != INF && ri.n_cells > 0 && l > 1e-6);
            deposit[i] = dep ? Q / l : 0.0;
        } else if (i < n) {
            deposit[i] = 0.0;                                         // outside the map's colony (MP with sizes)
        }
        const uint32_t ok = __ballot_sync(0xffffffffu, dep);
        if (lane == 0 && i < n) okbits[i >> 5] = ok;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double ol = __shfl_xor_sync(0xffffffffu, ml, o);
        const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
        if (lt_len_idx(ol, oi, ml, mi)) { ml = ol; mi = oi; }
    }
    if (lane == 0) { s_len[wid] = ml; s_idx[wid] = mi; }
    __syncthreads();
    if (wid == 0) {
        ml = s_len[lane]; mi = s_idx[lane];
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const double ol = __shfl_xor_sync(0xffffffffu, ml, o);
            const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
            if (lt_len_idx(ol, oi, ml, mi)) { ml = ol; mi = oi; }
        }
        if (lane == 0) { b_len = ml; b_r = mi; }
    }
    __syncthreads();
    const double L = b_len;
    const int r = b_r;
    // phase 2: among {r} U {i>r : |len_i - L| < 1e-9} the first index with the fewest turns
    int bt = 0x7fffffff, bi = 0x7fffffff;
    if (L != INF) {
        for (int i = tid; i < n_live; i += MPP_BEST_THREADS) {
            if (i < r) continue;
            const mpp_ant_result ri = res[i];
            const double l = ri.length;
            if (i == r || fabs(l - L) < 1e-9) {
                const int t = ri.turns;
                if (t >= 0 && (t < bt || (t == bt && i < bi))) { bt = t; bi = i; }
            }
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const int ot = __shfl_xor_sync(0xffffffffu, bt, o), oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ot < bt || (ot == bt && oi < bi)) { bt = ot; bi = oi; }
    }
    if (lane == 0) { s_t[wid] = bt; s_idx[wid] = bi; }
    __syncthreads();
    if (wid == 0) {
        bt = s_t[lane]; bi = s_idx[lane];
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const int ot = __shfl_xor_sync(0xffffffffu, bt, o), oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ot < bt || (ot == bt && oi < bi)) { bt = ot; bi = oi; }
        }
        if (lane == 0) {
            const bool any = (L != INF);
            b_ant = any ? bi : -1;
            b_turns = any ? bt : -1;
            // overall best MAACO.py:351-358
            mpp_maaco_state st = *state;
            int copy = 0;
            if (any) {
                if (L < st.best_len) {
                    st.best_len = L; st.best_turns = bt; copy = 1;
                } else if (fabs(L - st.best_len) < 1e-9) {
                    if (bt < st.best_turns) { st.best_turns = bt; copy = 1; }
                }
            }
            if (copy) { st.best_n_cells = res[bi].n_cells; st.best_iter = iteration; st.best_ant = bi; }
            st.iter_best_len = L; st.iter_best_turns = b_turns; st.iter_best_ant = b_ant;
            *state = st;
            b_copy = copy;
            if (log_all && iteration >= 1 && iteration <= log_rows) {
                double *lg = log_all + ((size_t)map * log_rows + (size_t)(iteration - 1)) * 4;
                lg[0] = L; lg[1] = (double)b_turns; lg[2] = st.best_len; lg[3] = (double)st.best_turns;
            }
        }
    }
    __syncthreads();
    // the path is decoded only by the rank that owns the ant (sharded colony: moves holds ants
    // [moves_ant_offset, moves_ant_offset + moves_n_ants)); the owner broadcasts it after the solve
    if (b_copy && b_ant >= moves_ant_offset && b_ant < moves_ant_offset + moves_n_ants) {
        const int a = b_ant - moves_ant_offset;
        int nm = res[b_ant].n_cells - 1;                             // moves of the path
        if (nm > max_cells) nm = max_cells;
        const uint8_t *mv = moves_all + ((size_t)map * moves_n_ants + a) * max_cells;
        int32_t *out = best_cells_all + (size_t)map * (max_cells + 1);
        if (tid == 0) { out[0] = meta[map].start; s_base = meta[map].start; }
        __syncthreads();
        for (int k0 = 0; k0 < nm; k0 += MPP_BEST_THREADS) {          // block-wide inclusive scan of the cell deltas
            const int k = k0 + tid;
            int x = (k < nm) ? move_delta(mv[k], C) : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
            if (lane == 31) s_idx[wid] = x;
            __syncthreads();
            if (wid == 0) {
                int w = s_idx[lane];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
                s_idx[lane] = w;
            }
            __syncthreads();
            const int cell = s_base + (wid ? s_idx[wid - 1] : 0) + x;
            if (k < nm) out[k + 1] = cell;
            __syncthreads();
            if (tid == MPP_BEST_THREADS - 1) s_base = cell;
            __syncthreads();
        }
    }
}
__global__ void __launch_bounds__(MPP_BEST_THREADS)
mpp_maaco_best_kernel(const mpp_ant_result *__restrict__ res_all, const uint8_t *__restrict__ moves_all, int max_cells,
                      int moves_ant_offset, int moves_n_ants, int n, double Q, int iteration, int C,
                      const MppMapMeta *__restrict__ meta, mpp_maaco_state *state_all, int32_t *best_cells_all,
                      double *deposit_all, uint32_t *okbits_all, double *log_all, int log_rows,
                      const int32_t *__restrict__ latch) {
    best_body<false>(res_all, moves_all, max_cells, moves_ant_offset, moves_n_ants, n, Q, nullptr, nullptr, iteration, C,
                     meta, state_all, best_cells_all, deposit_all, okbits_all, log_all, log_rows, latch);
}
__global__ void __launch_bounds__(MPP_BEST_THREADS)
mpp_maaco_best_p_kernel(const mpp_ant_result *__restrict__ res_all, const uint8_t *__restrict__ moves_all, int max_cells,
                        int moves_ant_offset, int moves_n_ants, int n, const mpp_maaco_params *__restrict__ params,
                        const int32_t *__restrict__ sizes, int iteration, int C, const MppMapMeta *__restrict__ meta,
                        mpp_maaco_state *state_all, int32_t *best_cells_all, double *deposit_all, uint32_t *okbits_all,
                        double *log_all, int log_rows, const int32_t *__restrict__ latch) {
    best_body<true>(res_all, moves_all, max_cells, moves_ant_offset, moves_n_ants, n, 0.0, params, sizes, iteration, C,
                    meta, state_all, best_cells_all, deposit_all, okbits_all, log_all, log_rows, latch);
}

static int best_launch(const mpp_map_batch *maps, const mpp_colony *c, int moves_ant_offset, int moves_n_ants,
                       int n_ants_total, double Q, const mpp_maaco_params *params_dev, int iteration, void *stream,
                       const int32_t *sizes_dev = nullptr) {
    int rc = colony_check(maps, c, "mpp_maaco_best");
    if (rc) return rc;
    MPP_REQUIRE(n_ants_total > 0 && iteration >= 1, "mpp_maaco_best: n_ants=%d iteration=%d", n_ants_total, iteration);
    MPP_CUDA(cudaSetDevice(maps->device));
    if (params_dev)
        mpp_maaco_best_p_kernel<<<maps->n_maps, MPP_BEST_THREADS, 0, (cudaStream_t)stream>>>(
            c->result, c->moves, c->max_cells, moves_ant_offset, moves_n_ants, n_ants_total, params_dev, sizes_dev,
            iteration, maps->cols, maps->meta_dev, c->state, c->best_cells, c->deposit, c->okbits, c->log, c->log_rows, c->latch);
    else
        mpp_maaco_best_kernel<<<maps->n_maps, MPP_BEST_THREADS, 0, (cudaStream_t)stream>>>(
            c->result, c->moves, c->max_cells, moves_ant_offset, moves_n_ants, n_ants_total, Q, iteration, maps->cols,
            maps->meta_dev, c->state, c->best_cells, c->deposit, c->okbits, c->log, c->log_rows, c->latch);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

extern "C" int mpp_maaco_best(const mpp_map_batch *maps, const mpp_colony *c, int moves_ant_offset, int moves_n_ants,
                              int n_ants_total, double Q, int iteration, void *stream) {
    return best_launch(maps, c, moves_ant_offset, moves_n_ants, n_ants_total, Q, nullptr, iteration, stream);
}

// ---------------------------------------------------------------------------------------------
// K3: pheromone evaporate + ordered deposit + MMAS clip (MAACO.py:304-332).
// One CTA per (map, tile, group of 8 tile rows); warp = one row of 32 cells, lane = cell.  The deposit of a cell
// is a sequential fp64 sum over the ants that visited it, in ant order (:306-311).  The CTA lists the ants that
// (a) have a slab for this tile (`touched`) and (b) deposit at all (`okbits`, from mpp_maaco_best) in index order and
// takes them 128 per trip: their 32-byte sectors (this row group's eight words) and their deposits go to shared
// memory with one 16-byte load per thread; each warp then takes its row 32 ants at a time, transposes the 32 x 32
// bit matrix (ant x cell) across its lanes and adds, per lane, the deposits of the ants that visited that lane's cell
// as a bare DADD chain (the operand is selected, t + 0.0 == t exactly).  Only slabs that exist are ever read: the
// traffic is 128 B per (ant, tile) pair + tau, not a dense bitmap.  (Details and measurements at the kernel.)
// ---------------------------------------------------------------------------------------------
#define MPP_PHER_THREADS 256
#define MPP_PHER_CHUNK 2048                   // ants per list-building round (64 bitmap words)
#define PHER_TRIP 128                         // ants the CTA takes per trip (256 threads x 16 bytes = their 32-byte sectors)
#define PHER_PITCH 132                        // row pitch of the shared-memory word tile (conflict-free transposing stores)

// MMAS clip + obstacle reset (MAACO.py:312-332) for one cell
__device__ __forceinline__ double pher_finalize(double t, int r, int c, const uint32_t *occ, int pitch, int R, int C,
                                                double rho, const mpp_maaco_state *state) {
    double b = state->best_len;                                               // :312-316
    if (b == __longlong_as_double(0x7ff0000000000000ll)) b = (double)(R + C);
    if (b < 1e-6) b = 1e-6;
    const double tmax = (1.0 / (1.0 - rho)) * (1.0 / b);                      // :317
    int mx = C > R ? C : R;
    if (mx < 1) mx = 1;
    const double tmin = tmax / (2.0 * (double)mx);                            // :323
    const int pb = c + 1;
    const bool obst = (occ[(r + 1) * pitch + (pb >> 5)] >> (pb & 31)) & 1u;
    if (obst) return 1e-9;                                                    // :332
    t = t > tmin ? t : tmin;                                                  // :327-331 np.clip
    return t < tmax ? t : tmax;
}

struct PherArgs {
    const uint32_t *occ; int occ_words, pitch, R, C;
    double *tau; size_t tau_stride;
    uint32_t *slabs; size_t slab_stride;        // [n_maps][buf tiles][n_ants][32]
    uint32_t *touched, *touched_next;           // this pass's bitmaps (read) / next pass's (cleared); [n_maps][buf tiles][NW]
    size_t touched_stride;
    const double *deposit; const uint32_t *okbits;
    int n_ants;                                 // all ants of the colony, global order
    int tile_row0;                              // first tile row of the buffers (a sharded colony updates a slice)
    double rho;
    const mpp_maaco_state *state;
    int clear_slabs;                            // zero the slab words that were read (sharded colony: rebuilt by OR next pass)
    const int32_t *latch;
    double *const *tau_peers; int n_peers;      // sharded colony over peer memory: every rank's tau (this rank's included)
    const MppMapMeta *meta;
};

#ifdef MPP_PHER_PROF
__device__ unsigned long long g_pher_prof[8192 * 8];
extern "C" int mpp_debug_pher_prof(unsigned long long *out) {
    return cudaMemcpyFromSymbol(out, g_pher_prof, sizeof(g_pher_prof)) == cudaSuccess ? 0 : -1;
}
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#endif

#ifndef MPP_PHER_MINB
#define MPP_PHER_MINB 7
#endif
// MP (per-map parameters): rho of params[map] instead of PherArgs' scalar; with sizes, a map past its pass count is left
// as it is (no evaporation).  Ants outside a map's colony have no `touched` and no `okbits` bits: nothing else changes.
template <bool MP>
__device__ __forceinline__ void pheromone_body(const PherArgs &A, const mpp_maaco_params *__restrict__ params,
                                               const int32_t *__restrict__ sizes, int iteration) {
    __shared__ int s_list[MPP_PHER_CHUNK];
#ifdef MPP_PHER_PROF
    const unsigned long long prof_t0 = gtimer();
    unsigned long long prof_hits = 0, prof_rounds = 0, prof_list = 0, prof_loop = 0, prof_tl = 0;
#endif
    __shared__ uint32_t s_w[2][8][PHER_PITCH];                        // a trip's row words [row of the group][ant], two trips
    __shared__ __align__(16) double s_d[2][PHER_TRIP];                // a trip's deposits
    __shared__ int s_wcnt[2];
    if (A.latch && *A.latch) return;
#ifdef MPP_PHER_ONLY
    if ((blockIdx.x >> 2) != MPP_PHER_ONLY) return;
#endif
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, map = blockIdx.y;
    double rho = A.rho;
    if constexpr (MP) {
        if (sizes && sized_past(sizes, map, iteration)) return;         // the whole CTA (grid.y = map)
        rho = params[map].rho;
    }
    const int TC = (A.C + 31) >> 5;
    // the start and the target tile carry the longest chains (every depositing ant): their CTAs go first
    int tile_l = blockIdx.x >> 2;                                     // tile index inside the buffers
    const int rg = blockIdx.x & 3;                                    // row group
    {
        const int nt = gridDim.x >> 2;
        const MppMapMeta &MM = A.meta[map];
        int h0 = ((MM.start / A.C >> 5) - A.tile_row0) * TC + (MM.start % A.C >> 5);
        int h1 = ((MM.target / A.C >> 5) - A.tile_row0) * TC + (MM.target % A.C >> 5);
        if (h0 < 0 || h0 >= nt) h0 = -1;
        if (h1 < 0 || h1 >= nt || h1 == h0) h1 = -1;
        if (h0 < 0) { h0 = h1; h1 = -1; }
        const int nh = (h0 >= 0) + (h1 >= 0);
        if (tile_l < nh) {
            tile_l = tile_l == 0 ? h0 : h1;
        } else {
            const int lo = (nh == 2 && h1 < h0) ? h1 : h0, hi = (nh == 2 && h1 < h0) ? h0 : h1;
            tile_l -= nh;
            if (nh >= 1 && tile_l >= lo) ++tile_l;
            if (nh == 2 && tile_l >= hi) ++tile_l;
        }
    }
    const int trow = A.tile_row0 + tile_l / TC, tcx = tile_l % TC;
    const int row_in_tile = rg * 8 + wid;
    const int r = (trow << 5) + row_in_tile, c = (tcx << 5) + lane;
    const bool live = r < A.R && c < A.C;
    double *tau = A.tau + (size_t)map * A.tau_stride;
    const int NW = (A.n_ants + 31) >> 5;
    const uint32_t *tb = A.touched + (size_t)map * A.touched_stride + (size_t)tile_l * NW;
    const uint32_t *ok = A.okbits + (size_t)map * NW;
    uint32_t *slab_t = A.slabs + (size_t)map * A.slab_stride + (size_t)tile_l * A.n_ants * 32 + row_in_tile;
    const double *dep = A.deposit + (size_t)map * A.n_ants;
    double t = 0.0;
    if (live) t = tau[(size_t)r * A.C + c] * (1.0 - rho);              // :305
    for (int w0 = 0; w0 < NW; w0 += MPP_PHER_CHUNK / 32) {
        // ---- the ants of this chunk that have a slab here and deposit, in index order ----
#ifdef MPP_PHER_PROF
        prof_tl = gtimer();
#endif
        int cnt = 0;
        uint32_t bits = 0u;
        if (wid < 2) {
            const int w = w0 + wid * 32 + lane;
            if (w < NW) bits = tb[w] & ok[w];
            cnt = __popc(bits);
            int x = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
            if (lane == 31) s_wcnt[wid] = x;
            cnt = x - cnt;                                             // exclusive prefix inside the warp
        }
        __syncthreads();
        const int k = s_wcnt[0] + s_wcnt[1];
        if (wid < 2) {
            int o = cnt + (wid ? s_wcnt[0] : 0);
            const int abase = (w0 + wid * 32 + lane) << 5;
            while (bits) { const int b = __ffs(bits) - 1; bits &= bits - 1; s_list[o++] = abase + b; }
        }
        __syncthreads();
#ifdef MPP_PHER_PROF
        { const unsigned long long g_ = gtimer(); prof_list += g_ - prof_tl; prof_tl = g_; }
#endif
        // ---- the rows.  The CTA takes 128 ants of the list per trip: thread t loads half of the 32-byte sector that holds
        //      this row group's eight words in ant t/2's slab (one 16-byte load: a warp load covers 16 lines, a per-row
        //      gather would cover 32 and repeat eight times) and threads 0..127 the deposits, both one trip ahead; they go
        //      to shared memory [row][ant] (double-buffered: one barrier per trip).  Then each warp folds ITS row: for every
        //      32 ants, lane i holds the row word of the i-th ant, the 32x32 bit matrix (ant x cell) is transposed across
        //      the warp so that lane c (= cell c of the row) holds the set of ants that visited its cell, and the lane adds
        //      the deposits of its own ants in index order (:306, :311).  Near the start and the target every ant crosses
        //      the same few cells, so some lane usually has all 32 bits set and 32 ants cost 32 dependent adds whatever
        //      the form: the fold is straight-line DADDs whose OPERAND is selected (t + 0.0 == t exactly; the
        //      loop-carried chain is the bare add, 8.2 cycles: tools/ubench/dadd_chain.cu), the deposits come from
        //      broadcast 16-byte shared-memory loads.  (tools/ubench/fold_round.cu, gather_round.cu: the forms that were
        //      tried -- compacted (word, deposit) lists with every lane adding every entry cost 27-36 cycles per add and
        //      ant, this 14; a per-warp gather costs 300 cycles of the SM's load path per 32 ants.) ----
        const int ntrip = (k + PHER_TRIP - 1) / PHER_TRIP;
        const uint32_t *slab_g = slab_t - wid + (threadIdx.x & 1) * 4;      // this row group's sector, this thread's half
        uint4 wv = make_uint4(0u, 0u, 0u, 0u);
        double dv = 0.0;
        int av = -1;
        auto issue = [&](int trip) {
            const int i = trip * PHER_TRIP + (threadIdx.x >> 1);
            wv = make_uint4(0u, 0u, 0u, 0u); av = -1; dv = 0.0;
            if (i < k) { av = s_list[i]; wv = *(const uint4 *)(slab_g + (size_t)av * 32); }
            if (threadIdx.x < PHER_TRIP) {
                const int i2 = trip * PHER_TRIP + threadIdx.x;
                if (i2 < k) dv = dep[s_list[i2]];
            }
        };
        issue(0);
        for (int trip = 0; trip < ntrip; ++trip) {
            const int buf = trip & 1;
            {
                uint32_t *dst = &s_w[buf][(threadIdx.x & 1) * 4][threadIdx.x >> 1];
                dst[0] = wv.x; dst[PHER_PITCH] = wv.y; dst[2 * PHER_PITCH] = wv.z; dst[3 * PHER_PITCH] = wv.w;
                if (threadIdx.x < PHER_TRIP) s_d[buf][threadIdx.x] = dv;
                if (A.clear_slabs && (wv.x | wv.y | wv.z | wv.w)) *(uint4 *)(const_cast<uint32_t *>(slab_g) + (size_t)av * 32) = make_uint4(0u, 0u, 0u, 0u);
            }
            issue(trip + 1);                                           // in flight while this trip is folded
            __syncthreads();
#pragma unroll 1
            for (int r = 0; r < PHER_TRIP / 32; ++r) {
                if (trip * PHER_TRIP + r * 32 >= k) break;
                uint32_t m = s_w[buf][wid][r * 32 + lane];
                const uint32_t nz = __ballot_sync(0xffffffffu, m != 0u);
                if (!nz) continue;
#ifdef MPP_PHER_PROF
                prof_hits += __popc(nz); prof_rounds += 1;
#endif
#pragma unroll
                for (int j = 16, mk = 0x0000FFFF; j; j >>= 1, mk ^= mk << j) {
                    const uint32_t y = __shfl_xor_sync(0xffffffffu, m, j);
                    m = (lane & j) ? ((m & ~(uint32_t)mk) | ((y >> j) & (uint32_t)mk)) : ((m & (uint32_t)mk) | ((y << j) & ~(uint32_t)mk));
                }
                const double2 *sd2 = (const double2 *)(s_d[buf] + r * 32);
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    if (!(nz & (0xFFu << (8 * g)))) continue;          // (warp-uniform) none of these eight ants has a word here
                    const double2 v0 = sd2[4 * g], v1 = sd2[4 * g + 1], v2 = sd2[4 * g + 2], v3 = sd2[4 * g + 3];
                    const uint32_t mg = m >> (8 * g);
                    // (the operand is selected, not the sum: the loop-carried chain is a bare DADD; t + 0.0 == t exactly)
                    const double a0 = (mg & 1u) ? v0.x : 0.0, a1 = (mg & 2u) ? v0.y : 0.0, a2 = (mg & 4u) ? v1.x : 0.0;
                    const double a3 = (mg & 8u) ? v1.y : 0.0, a4 = (mg & 16u) ? v2.x : 0.0, a5 = (mg & 32u) ? v2.y : 0.0;
                    const double a6 = (mg & 64u) ? v3.x : 0.0, a7 = (mg & 128u) ? v3.y : 0.0;
                    t += a0;
                    t += a1;
                    t += a2;
                    t += a3;
                    t += a4;
                    t += a5;
                    t += a6;
                    t += a7;
                }
            }
        }
#ifdef MPP_PHER_PROF
        prof_loop += gtimer() - prof_tl;
#endif
        __syncthreads();                                               // s_list is rebuilt by the next chunk
    }
    if (live) {
        const double v = pher_finalize(t, r, c, A.occ + (size_t)map * A.occ_words, A.pitch, A.R, A.C, rho, A.state + map);
        if (A.tau_peers) {
            // fused with the "all-gather" of the tau slices: the value goes straight into every rank's field (NVLink stores)
            for (int k = 0; k < A.n_peers; ++k) A.tau_peers[k][(size_t)r * A.C + c] = v;
        } else {
            tau[(size_t)r * A.C + c] = v;
        }
    }
#ifdef MPP_PHER_PROF
    if (lane == 0 && blockIdx.y == 0 && blockIdx.x * 8 + wid < 8192) {
        unsigned long long *o = g_pher_prof + (size_t)(blockIdx.x * 8 + wid) * 8;
        o[0] = prof_t0; o[1] = gtimer(); o[2] = prof_hits; o[3] = prof_rounds;
        o[4] = prof_list; o[5] = prof_loop; o[6] = o[7] = 0;
    }
#endif
    // the bitmaps the NEXT pass will fill are the ones the previous pass consumed: clear this tile's share
    {
        uint32_t *tn = A.touched_next + (size_t)map * A.touched_stride + (size_t)tile_l * NW;
        for (int w = rg * MPP_PHER_THREADS + threadIdx.x; w < NW; w += 4 * MPP_PHER_THREADS) tn[w] = 0u;
    }
}
__global__ void __launch_bounds__(MPP_PHER_THREADS, MPP_PHER_MINB) mpp_maaco_pheromone_kernel(const PherArgs A) {
    pheromone_body<false>(A, nullptr, nullptr, 0);
}
__global__ void __launch_bounds__(MPP_PHER_THREADS, MPP_PHER_MINB)
mpp_maaco_pheromone_p_kernel(const PherArgs A, const mpp_maaco_params *__restrict__ params,
                             const int32_t *__restrict__ sizes, int iteration) {
    pheromone_body<true>(A, params, sizes, iteration);
}

static int pheromone_launch(const mpp_map_batch *maps, const mpp_colony *c, uint32_t *slabs_dev, uint32_t *touched_dev,
                            int n_ants_total, int tile_row0, int buf_tile_rows, double rho, int iteration, int clear_slabs,
                            double *const *tau_peers_dev, int n_peers, void *stream,
                            const mpp_maaco_params *params_dev = nullptr, const int32_t *sizes_dev = nullptr) {
    int rc = colony_check(maps, c, "mpp_maaco_pheromone");
    if (rc) return rc;
    const int TR = tiles_r(maps->rows), TC = tiles_c(maps->cols);
    MPP_REQUIRE(slabs_dev && touched_dev && n_ants_total > 0, "mpp_maaco_pheromone: null argument");
    MPP_REQUIRE(tile_row0 >= 0 && buf_tile_rows > 0, "mpp_maaco_pheromone: bad tile-row range");
    MPP_CUDA(cudaSetDevice(maps->device));
    int n_tile_rows = buf_tile_rows;                                  // rows of the buffers that lie inside the map
    if (tile_row0 + n_tile_rows > TR) n_tile_rows = TR - tile_row0;
    if (n_tile_rows <= 0) return MPP_OK;                              // a padded slice beyond the map
    const int NW = (n_ants_total + 31) / 32;
    PherArgs A;
    A.occ = maps->occ_dev; A.occ_words = maps->occ_words; A.pitch = maps->pitch_words; A.R = maps->rows; A.C = maps->cols;
    A.tau = c->tau; A.tau_stride = (size_t)c->tau_stride;
    A.slabs = slabs_dev;
    A.slab_stride = (size_t)buf_tile_rows * TC * (size_t)n_ants_total * 32;
    A.touched_stride = (size_t)buf_tile_rows * TC * (size_t)NW;
    const size_t par = A.touched_stride * maps->n_maps;
    A.touched = touched_dev + (size_t)(iteration & 1) * par;
    A.touched_next = touched_dev + (size_t)((iteration + 1) & 1) * par;
    A.deposit = c->deposit; A.okbits = c->okbits; A.n_ants = n_ants_total;
    A.tile_row0 = tile_row0; A.rho = rho; A.state = c->state; A.clear_slabs = clear_slabs;
    A.latch = c->latch;
    A.tau_peers = tau_peers_dev; A.n_peers = n_peers;
    A.meta = maps->meta_dev;
    MPP_REQUIRE(!tau_peers_dev || (n_peers > 0 && maps->n_maps == 1), "mpp_maaco_pheromone: peer tau needs n_peers > 0 and one map");
    const dim3 grid(n_tile_rows * TC * 4, maps->n_maps);
    if (params_dev)
        mpp_maaco_pheromone_p_kernel<<<grid, MPP_PHER_THREADS, 0, (cudaStream_t)stream>>>(A, params_dev, sizes_dev, iteration);
    else mpp_maaco_pheromone_kernel<<<grid, MPP_PHER_THREADS, 0, (cudaStream_t)stream>>>(A);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

extern "C" int mpp_maaco_pheromone(const mpp_map_batch *maps, const mpp_colony *c, uint32_t *slabs_dev, uint32_t *touched_dev,
                                   int n_ants_total, int tile_row0, int buf_tile_rows, double rho, int iteration,
                                   int clear_slabs, double *const *tau_peers_dev, int n_peers, void *stream) {
    return pheromone_launch(maps, c, slabs_dev, touched_dev, n_ants_total, tile_row0, buf_tile_rows, rho, iteration,
                            clear_slabs, tau_peers_dev, n_peers, stream);
}

// ---------------------------------------------------------------------------------------------
// Sharded-colony exchange, all-gather form (the fallback: with NVLink peer access the tour kernel's P2P instantiation
// delivers slabs and results itself, mpp_maaco_tours_p2p, and none of this runs).  Rank g constructs its ants and ships
// (a) their 16-byte results and (b) their tours as 1-byte move codes in ONE buffer per pass (one all-gather); every rank
// then replays the codes of all ants into slabs of ITS slice of tile rows and updates the pheromone of that slice with all
// ants in global order.
//   exchange buffer of one rank: [n_local x mpp_ant_result][int32 total code bytes, 3 x int32 pad][codes ...]
// ---------------------------------------------------------------------------------------------
#define MPP_XHDR(n_local) ((size_t)16 * (size_t)(n_local) + 16)

// exclusive scan of (n_cells - 1, 0 for failed ants) over one segment's results; one block of 1024 threads.
// offsets[a] = byte offset of ant a's codes; returns the total through *total_out.
__device__ __forceinline__ void xscan_segment(const mpp_ant_result *__restrict__ res, int seg_ants, int32_t *__restrict__ offsets,
                                              int *s_warp, int *s_carry, int *total_out) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) *s_carry = 0;
    __syncthreads();
    for (int base = 0; base < seg_ants; base += 1024) {
        const int a = base + tid;
        int len = 0;
        if (a < seg_ants) { const int n = res[a].n_cells; len = n > 0 ? n - 1 : 0; }
        int x = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        if (lane == 31) s_warp[wid] = x;
        __syncthreads();
        if (wid == 0) {
            int w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
            s_warp[lane] = w;
        }
        __syncthreads();
        const int excl = *s_carry + (wid ? s_warp[wid - 1] : 0) + x - len;
        if (a < seg_ants) offsets[a] = excl;
        __syncthreads();
        if (tid == 1023) *s_carry += s_warp[31];
        __syncthreads();
    }
    *total_out = *s_carry;
}

// step 1 on the sending rank: header (results + total) and the offsets of the local ants
// (peers != null: the buffer is written straight into slot `peer_off` of every rank's receive buffer -- the
// "all-gather" fused into the producer over NVLink peer memory; peers == null: into this rank's send buffer xbuf)
__global__ void __launch_bounds__(1024) mpp_maaco_xpack_scan_kernel(const mpp_ant_result *__restrict__ res_local, int n_local,
                                                                    int32_t *__restrict__ offsets_local, uint8_t *__restrict__ xbuf,
                                                                    uint8_t *const *__restrict__ peers, int n_peers, size_t peer_off,
                                                                    const int32_t *__restrict__ latch) {
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    if (latch && *latch) return;
    int total;
    xscan_segment(res_local, n_local, offsets_local, s_warp, &s_carry, &total);
    const int nd = peers ? n_peers : 1;
    for (int k = 0; k < nd; ++k) {
        uint8_t *dst = peers ? peers[k] + peer_off : xbuf;
        mpp_ant_result *hdr = (mpp_ant_result *)dst;
        for (int a = threadIdx.x; a < n_local; a += 1024) hdr[a] = res_local[a];
        if (threadIdx.x == 0) {
            int32_t *tail = (int32_t *)(dst + (size_t)16 * n_local);
            tail[0] = total; tail[1] = 0; tail[2] = 0; tail[3] = 0;
        }
    }
}

// step 2: one warp per local ant copies its move codes behind the header (nothing is written past `cap`; the
// receivers see total > cap in the header and raise the latch)
__global__ void __launch_bounds__(256) mpp_maaco_xpack_copy_kernel(const uint8_t *__restrict__ moves, int max_cells,
                                                                   const mpp_ant_result *__restrict__ res_local,
                                                                   const int32_t *__restrict__ offsets_local, int n_local,
                                                                   uint8_t *__restrict__ xbuf, long long cap,
                                                                   uint8_t *const *__restrict__ peers, int n_peers, size_t peer_off,
                                                                   const int32_t *__restrict__ latch) {
    if (latch && *latch) return;
    const int a = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (a >= n_local) return;
    const int n = res_local[a].n_cells;
    if (n <= 1) return;
    const long long off = offsets_local[a];
    if (n - 1 > max_cells || off + (n - 1) > cap) return;
    const uint8_t *src = moves + (size_t)a * max_cells;
    const int nd = peers ? n_peers : 1;
    for (int i = lane; i < n - 1; i += 32) {
        const uint8_t v = src[i];
        for (int k = 0; k < nd; ++k) ((peers ? peers[k] + peer_off : xbuf) + MPP_XHDR(n_local) + off)[i] = v;
    }
}

// step 3 on every rank after the all-gather: results of all segments into the contiguous table, per-ant code offsets,
// overflow check (a tour longer than max_cells or a segment larger than `cap` raises the latch = this iteration),
// and the clearing of the local `touched` bitmaps of the NEXT pass (nobody consumes a sharded rank's own slabs)
__global__ void __launch_bounds__(1024) mpp_maaco_xunpack_kernel(const uint8_t *__restrict__ xbuf_all, size_t seg_stride,
                                                                 int seg_ants, long long cap, int max_cells,
                                                                 mpp_ant_result *__restrict__ result,
                                                                 int32_t *__restrict__ offsets, int32_t *latch, int iteration,
                                                                 uint32_t *__restrict__ clear_ptr, size_t clear_words) {
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    __shared__ int s_long;
    if (*latch) return;
    const int seg = blockIdx.x;
    const uint8_t *xb = xbuf_all + (size_t)seg * seg_stride;
    const mpp_ant_result *hdr = (const mpp_ant_result *)xb;
    if (threadIdx.x == 0) s_long = 0;
    int total;
    xscan_segment(hdr, seg_ants, offsets + (size_t)seg * seg_ants, s_warp, &s_carry, &total);
    for (int a = threadIdx.x; a < seg_ants; a += 1024) {
        const mpp_ant_result r = hdr[a];
        result[(size_t)seg * seg_ants + a] = r;
        if (r.n_cells - 1 > max_cells) s_long = 1;
    }
    for (size_t w = (size_t)seg * 1024 + threadIdx.x; w < clear_words; w += (size_t)gridDim.x * 1024) clear_ptr[w] = 0u;
    __syncthreads();
    if (threadIdx.x == 0 && (total > cap || s_long)) atomicMax(latch, iteration);
}

// step 4: one warp per global ant replays its moves 32 at a time (warp prefix sum of the cell deltas) and sets the
// visited bits that fall into tile rows [tile_row0, tile_row0 + buf_tile_rows) of the receive slabs
// ([tile][all ants][32], zero on entry: the update clears what it reads) and the (tile, ant) bits of `touched`.
__global__ void __launch_bounds__(256) mpp_maaco_rebuild_kernel(const uint8_t *__restrict__ xbuf_all, size_t seg_stride,
                                                                const int32_t *__restrict__ offsets,
                                                                const mpp_ant_result *__restrict__ res, int n_seg,
                                                                int seg_ants, int start, int C, int TC, int tile_row0,
                                                                int buf_tile_rows, uint32_t *__restrict__ slabs,
                                                                uint32_t *__restrict__ touched,
                                                                const int32_t *__restrict__ latch) {
    if (*latch) return;
    const int g = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int n_total = n_seg * seg_ants;
    if (g >= n_total) return;
    const int n = res[g].n_cells;
    if (n <= 0) return;                                      // failed ants deposit nothing (MAACO.py:307)
    const int seg = g / seg_ants;
    const uint8_t *codes = xbuf_all + (size_t)seg * seg_stride + MPP_XHDR(seg_ants) + offsets[g];
    const int NW = (n_total + 31) >> 5;
    auto mark = [&](int cell, bool first_of_tile) {
        const int r = cell / C, c = cell - r * C;
        const int trl = (r >> 5) - tile_row0;
        if (trl < 0 || trl >= buf_tile_rows) return;
        const int tile_l = trl * TC + (c >> 5);
        atomicOr(slabs + ((size_t)tile_l * n_total + g) * 32 + (r & 31), 1u << (c & 31));
        if (first_of_tile) atomicOr(touched + (size_t)tile_l * NW + (g >> 5), 1u << (g & 31));
    };
    int base_cell = start;                                   // cell before the first move of the current chunk
    if (lane == 0) mark(start, true);
    for (int i0 = 0; i0 < n - 1; i0 += 32) {
        const int i = i0 + lane;
        int d = 0;
        if (i < n - 1) d = move_delta(codes[i], C);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, d, o); if (lane >= o) d += y; }
        const int cell = base_cell + d;                      // cell reached after move i
        // (tile, ant) bit: once per run of cells inside one tile (the lane before is in another tile, or lane 0)
        const int tkey = ((cell / C) >> 5) * TC + ((cell % C) >> 5);
        const int tprev = __shfl_up_sync(0xffffffffu, tkey, 1);
        if (i < n - 1) mark(cell, lane == 0 || tprev != tkey);
        base_cell = __shfl_sync(0xffffffffu, cell, 31);
    }
}

extern "C" long long mpp_maaco_xhdr_bytes(int n_local) { return (long long)MPP_XHDR(n_local); }

extern "C" int mpp_maaco_xpack(const mpp_map_batch *maps, const mpp_colony *c, int ant_offset, int n_local, int n_ants_total,
                               int32_t *offsets_local_dev, uint8_t *xbuf_local_dev, long long capacity,
                               uint8_t *const *peer_xbuf_dev, int n_peers, int rank, void *stream) {
    int rc = colony_check(maps, c, "mpp_maaco_xpack");
    if (rc) return rc;
    MPP_REQUIRE(maps->n_maps == 1, "mpp_maaco_xpack: a sharded colony is one map");
    MPP_REQUIRE(offsets_local_dev && (xbuf_local_dev || peer_xbuf_dev) && n_local > 0 && capacity >= 0 &&
                    ant_offset + n_local <= n_ants_total, "mpp_maaco_xpack: bad argument");
    MPP_REQUIRE(!peer_xbuf_dev || (n_peers > 0 && rank >= 0 && rank < n_peers), "mpp_maaco_xpack: bad peer arguments");
    const size_t peer_off = (size_t)rank * (MPP_XHDR(n_local) + (size_t)capacity);   // this rank's slot in every receive buffer
    MPP_CUDA(cudaSetDevice(maps->device));
    cudaStream_t s = (cudaStream_t)stream;
    mpp_maaco_xpack_scan_kernel<<<1, 1024, 0, s>>>(c->result + ant_offset, n_local, offsets_local_dev, xbuf_local_dev,
                                                   peer_xbuf_dev, n_peers, peer_off, c->latch);
    mpp_maaco_xpack_copy_kernel<<<(n_local + 7) / 8, 256, 0, s>>>(c->moves, c->max_cells, c->result + ant_offset,
                                                                  offsets_local_dev, n_local, xbuf_local_dev, capacity,
                                                                  peer_xbuf_dev, n_peers, peer_off, c->latch);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

extern "C" int mpp_maaco_xunpack(const mpp_map_batch *maps, const mpp_colony *c, const uint8_t *xbuf_all_dev, long long capacity,
                                 int n_seg, int seg_ants, int iteration, int32_t *offsets_dev, int tile_row0, int buf_tile_rows,
                                 uint32_t *slabs_recv_dev, uint32_t *touched_recv_dev, uint32_t *touched_local_dev,
                                 void *stream) {
    int rc = colony_check(maps, c, "mpp_maaco_xunpack");
    if (rc) return rc;
    MPP_REQUIRE(maps->n_maps == 1, "mpp_maaco_xunpack: a sharded colony is one map");
    MPP_REQUIRE(xbuf_all_dev && offsets_dev && slabs_recv_dev && touched_recv_dev && touched_local_dev && c->latch &&
                    n_seg > 0 && seg_ants > 0 && capacity >= 0, "mpp_maaco_xunpack: bad argument");
    MPP_CUDA(cudaSetDevice(maps->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int TR = tiles_r(maps->rows), TC = tiles_c(maps->cols);
    const size_t seg_stride = MPP_XHDR(seg_ants) + (size_t)capacity;
    const int n_total = n_seg * seg_ants;
    // the local tour buffers of the next pass: parity (iteration + 1)
    const size_t tw_local = (size_t)mpp_maaco_touched_words(TR, maps->cols, seg_ants) / 2;
    uint32_t *clear_ptr = touched_local_dev + (size_t)((iteration + 1) & 1) * tw_local;
    mpp_maaco_xunpack_kernel<<<n_seg, 1024, 0, s>>>(xbuf_all_dev, seg_stride, seg_ants, capacity, c->max_cells, c->result,
                                                    offsets_dev, (int32_t *)c->latch, iteration, clear_ptr, tw_local);
    const size_t tw_recv = (size_t)mpp_maaco_touched_words(buf_tile_rows, maps->cols, n_total) / 2;
    mpp_maaco_rebuild_kernel<<<(n_total + 7) / 8, 256, 0, s>>>(
        xbuf_all_dev, seg_stride, offsets_dev, c->result, n_seg, seg_ants, maps->meta_host[0].start, maps->cols, TC,
        tile_row0, buf_tile_rows, slabs_recv_dev, touched_recv_dev + (size_t)(iteration & 1) * tw_recv, c->latch);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

// ---------------------------------------------------------------------------------------------
// One whole colony pass of a non-sharded colony (ranking, tours, best tracking, pheromone update), and the same
// pass driven with HOST buffers: the pheromone field goes in, the per-ant results, the colony state, the best path
// and the updated field come out, all inside the call (the reference-facing, synchronous form of the hot path).
// ---------------------------------------------------------------------------------------------
extern "C" int mpp_maaco_pass(const mpp_map_batch *maps, const mpp_colony *c, const mpp_maaco_params *p, int iteration,
                              int n_ants, int ants_per_warp, void *stream) {
    MPP_REQUIRE(p, "mpp_maaco_pass: null params");
    int rc = mpp_maaco_rank(maps, c, p->alpha, stream);
    if (rc) return rc;
    rc = mpp_maaco_tours(maps, c, iteration, mpp_maaco_q0(p->num_iterations, iteration, p->q0_initial), p->alpha, n_ants, 0,
                         n_ants, ants_per_warp, stream);
    if (rc) return rc;
    rc = mpp_maaco_best(maps, c, 0, n_ants, n_ants, p->Q, iteration, stream);
    if (rc) return rc;
    return mpp_maaco_pheromone(maps, c, c->slabs, c->touched, n_ants, 0, tiles_r(maps->rows), p->rho, iteration, 0, nullptr, 0, stream);
}

// The same pass with per-map colony parameters: params_dev [n_maps] on the device, q0_dev the [num_iterations][n_maps]
// q0 table (row iteration-1 is this pass's); the per-map instantiations of the four kernels read their scalars from them.
// sizes_dev (null, or [n_maps] {num_ants, num_iterations} on the device) gives each map its own colony inside the
// buffers' n_ants and its own pass count (sized_ants / sized_past).
extern "C" int mpp_maaco_pass_maps_sized(const mpp_map_batch *maps, const mpp_colony *c, const mpp_maaco_params *params_dev,
                                         const double *q0_dev, const int32_t *sizes_dev, int iteration, int n_ants,
                                         int ants_per_warp, void *stream) {
    MPP_REQUIRE(maps && c, "mpp_maaco_pass_maps: null argument");
    MPP_REQUIRE(params_dev && q0_dev, "mpp_maaco_pass_maps: null params_dev / q0_dev");
    MPP_REQUIRE(iteration >= 1, "mpp_maaco_pass_maps: iteration %d < 1", iteration);
    int rc = rank_launch(maps, c, 0.0, params_dev, stream, sizes_dev, iteration);
    if (rc) return rc;
    const TourMapParams mp{params_dev, q0_dev + (size_t)(iteration - 1) * maps->n_maps, sizes_dev};
    rc = tours_launch(maps, c, iteration, 0.0, 0.0, n_ants, 0, n_ants, ants_per_warp, nullptr, nullptr, nullptr, 0, 1, stream,
                      &mp);
    if (rc) return rc;
    rc = best_launch(maps, c, 0, n_ants, n_ants, 0.0, params_dev, iteration, stream, sizes_dev);
    if (rc) return rc;
    return pheromone_launch(maps, c, c->slabs, c->touched, n_ants, 0, tiles_r(maps->rows), 0.0, iteration, 0, nullptr, 0,
                            stream, params_dev, sizes_dev);
}

extern "C" int mpp_maaco_pass_maps(const mpp_map_batch *maps, const mpp_colony *c, const mpp_maaco_params *params_dev,
                                   const double *q0_dev, int iteration, int n_ants, int ants_per_warp, void *stream) {
    return mpp_maaco_pass_maps_sized(maps, c, params_dev, q0_dev, nullptr, iteration, n_ants, ants_per_warp, stream);
}

extern "C" int mpp_maaco_pass_host(const mpp_map_batch *maps, const mpp_colony *c, const mpp_maaco_params *p, int iteration,
                                   int n_ants, int ants_per_warp, const double *tau_in_host, double *tau_out_host,
                                   mpp_ant_result *result_out_host, mpp_maaco_state *state_out_host,
                                   int32_t *best_cells_out_host, int best_cells_capacity, void *stream) {
    int rc = colony_check(maps, c, "mpp_maaco_pass_host");
    if (rc) return rc;
    MPP_CUDA(cudaSetDevice(maps->device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)maps->rows * maps->cols;
    const int M = maps->n_maps;
    if (tau_in_host)
        MPP_CUDA(cudaMemcpy2DAsync(c->tau, (size_t)c->tau_stride * 8, tau_in_host, n * 8, n * 8, M, cudaMemcpyHostToDevice, s));
    rc = mpp_maaco_pass(maps, c, p, iteration, n_ants, ants_per_warp, stream);
    if (rc) return rc;
    if (tau_out_host)
        MPP_CUDA(cudaMemcpy2DAsync(tau_out_host, n * 8, c->tau, (size_t)c->tau_stride * 8, n * 8, M, cudaMemcpyDeviceToHost, s));
    if (result_out_host)
        MPP_CUDA(cudaMemcpyAsync(result_out_host, c->result, sizeof(mpp_ant_result) * (size_t)n_ants * M, cudaMemcpyDeviceToHost, s));
    if (state_out_host)
        MPP_CUDA(cudaMemcpyAsync(state_out_host, c->state, sizeof(mpp_maaco_state) * M, cudaMemcpyDeviceToHost, s));
    if (best_cells_out_host) {
        int cap = best_cells_capacity < c->max_cells + 1 ? best_cells_capacity : c->max_cells + 1;
        MPP_CUDA(cudaMemcpy2DAsync(best_cells_out_host, (size_t)best_cells_capacity * 4, c->best_cells, (size_t)(c->max_cells + 1) * 4,
                                   (size_t)cap * 4, M, cudaMemcpyDeviceToHost, s));
    }
    MPP_CUDA(cudaStreamSynchronize(s));
    return MPP_OK;
}
