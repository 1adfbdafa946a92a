/*
 * mpp.h -- C ABI of libmpp_b200.so: the B200 (sm_100a) implementation of the
 * population-evaluation hot path of dvnam1605/MAACO-path-planing.
 *
 * The reference has no FFI of its own (pure Python); this header is the boundary a
 * maintainer binds with ctypes underneath the reference's Python classes (see
 * INTEGRATION.md for the stub).  Each entry point names the reference code it
 * replaces (file:line relative to the reference tree).
 *
 * Conventions
 *   - every function returns 0 on success, a negative MPP_E* code otherwise; nothing
 *     throws across the ABI; mpp_last_error() returns a thread-local message.
 *   - all pointers named *_dev are device pointers on the map's device; everything is
 *     enqueued on `stream` (a cudaStream_t passed as void*) and is asynchronous unless
 *     stated.  The caller owns every buffer; the library owns only map handles.
 *   - cells are int32 `r*cols + c`; paths are int32 arrays; all reals are IEEE binary64.
 *   - there is NO CPU fallback: with no sm_100 device the calls fail with MPP_ENODEVICE.
 *   - RNG: counter-based Philox4x32-10 streams keyed (seed, class, iteration, individual)
 *     with an in-stream cursor (DESIGN.md "RNG contract").
 */
#ifndef MPP_H_
#define MPP_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPP_ABI_VERSION 3

#define MPP_OK 0
#define MPP_EINVAL (-1)
#define MPP_ENODEVICE (-2)
#define MPP_ECUDA (-3)
#define MPP_ENOMEM (-4)
#define MPP_EUNSUPPORTED (-5)

/* stream classes of the RNG contract */
#define MPP_CLS_MAACO_TOUR 1
#define MPP_CLS_PSO_INIT 2
#define MPP_CLS_PSO_PAD 3
#define MPP_CLS_PSO_UPDATE 4
#define MPP_CLS_GA_INIT 5
#define MPP_CLS_GA_PAD 6
#define MPP_CLS_GA_SELECT 7
#define MPP_CLS_GA_BREED 8
#define MPP_CLS_MPA_PHASE 9
#define MPP_CLS_MPA_FADS 10

int mpp_abi_version(void);
const char *mpp_last_error(void);
/* number of sm_100 devices visible (0 => every compute entry point fails) */
int mpp_device_count(void);

/* ---- maps: env.py grid convention (0 free, 1 obstacle, 2 start, 3 target) -------------------------------------------
 * A batch of independent same-shape maps (BASELINE config 5: "batched sweep over independent maps") on one device; every
 * compute entry point takes a batch, and a single map is a batch of one (n_maps = 1).
 * replaces: np.array(grid) + argwhere(grid==2/3) in every constructor
 * (MAACO.py:15-41, helper.py:121-125, astar.py:17-22, pso.py:17-22, ga_solver.py:17-22, MPA.py:20-43), and a Python loop
 * `for grid in grids: MAACO(grid, ...)` around MAACO.py:11-53.
 * grids_host: n_maps x rows x cols bytes, row-major.  Start/target of a map = its first row-major 2 / 3.  Synchronous. */
typedef struct mpp_map_batch mpp_map_batch; /* opaque: bit-packed occupancy grids + per-map tables on one device */
int mpp_map_batch_create(const uint8_t *grids_host, int n_maps, int rows, int cols, int device, mpp_map_batch **out);
void mpp_map_batch_destroy(mpp_map_batch *maps);
int mpp_map_batch_size(const mpp_map_batch *maps);
int mpp_map_batch_start(const mpp_map_batch *maps, int k);  /* cell id of map k's start or -1 */
int mpp_map_batch_target(const mpp_map_batch *maps, int k);
/* The same batch from grids already in device memory of `device`: grids_dev = n_maps x rows x cols contiguous cells of
 * elem_bytes bytes each (1 = uint8, 4 = int32, 8 = int64).  Cells are compared raw: 1 obstacle, 2 start candidate,
 * 3 target candidate, any other value free -- the classification the uint8 path gives after clipping to 0..255.
 * Everything runs on `stream` (the grids may have been written by work enqueued on it just before); the grids never
 * leave the device, only the per-map start / target and the obstacle count are read back.  Synchronous: returns when
 * the batch is ready. */
int mpp_map_batch_create_device(const void *grids_dev, int elem_bytes, int n_maps, int rows, int cols, int device,
                                void *stream, mpp_map_batch **out);
/* the batch's occupancy, [n_maps][((rows+2) * pitch_words + 3) & ~3] words: border-padded and bit-packed, bit (r+1, c+1)
 * of map k in row r+1 of its slice (pitch_words 32-bit words per row), the border marked occupied; its static move masks
 * [n_maps][rows*cols] (MAACO move order) and its obstacle count over all maps */
const uint32_t *mpp_map_batch_occ_bits(const mpp_map_batch *maps, int *pitch_words);
const uint8_t *mpp_map_batch_svalid(const mpp_map_batch *maps);
long long mpp_map_batch_obstacles(const mpp_map_batch *maps);

/* ---- MAACO (MAACO.py) -------------------------------------------------------------------- */
typedef struct {
    double alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min, k_h_adaptive, q0_initial, C0_initial_pheromone;
    int num_iterations;
} mpp_maaco_params;

/* per-ant outcome of one tour (MAACO.py:300-302): failed ants have n_cells=0, length=+inf, turns=-1 */
typedef struct {
    double length;
    int32_t n_cells;
    int32_t turns;
} mpp_ant_result;

/* colony state kept on the device so an entire solve can be enqueued without host syncs */
typedef struct {
    double best_len;       /* best_path_length_overall (+inf = none) */
    int32_t best_turns;    /* -1 = inf */
    int32_t best_n_cells;
    int32_t best_iter;     /* iteration that set best_path (0 = none) */
    int32_t best_ant;
    double iter_best_len;  /* last iteration */
    int32_t iter_best_turns;
    int32_t iter_best_ant; /* -1 = all ants failed */
} mpp_maaco_state;

/* The device buffers of a colony (or of one colony per map of a batch), all owned by the caller.  n_ants below is
 * the number of ants THIS process constructs per map (a sharded colony: its shard), n_total the colony size.
 * TR = ceil(rows/32), TC = ceil(cols/32): the map as tiles of 32 x 32 cells. */
typedef struct {
    double *tau;               /* [n_maps][tau_stride] pheromone field (MAACO.pheromone_matrix), tau_stride >= rows*cols */
    long long tau_stride;
    const double *E01;         /* [n_maps or 1][2*rows*cols] eta'**beta by turn flag, interleaved (mpp_maaco_tables) */
    long long E01_stride;      /* 0 = one table shared by every map of the batch */
    uint32_t *rank;            /* [n_maps][mpp_maaco_rank_words(rows, cols)] (mpp_maaco_rank) */
    uint32_t *slabs;           /* [n_maps][TR*TC][n_ants][32]: visited bits of one ant inside one tile, a word per tile row;
                                  mpp_maaco_slab_words(TR, cols, n_ants) words per map.  Never needs clearing. */
    uint32_t *touched;         /* [2][n_maps][TR*TC][ceil(n_ants/32)]: (tile, ant) has a slab this pass, double buffered by
                                  iteration parity; mpp_maaco_touched_words(TR, cols, n_ants) words per map; zero before the
                                  first pass (the pheromone update keeps clearing the buffer of the next pass) */
    uint8_t *moves;            /* [n_maps][n_ants][max_cells] tours as move codes (move order MAACO.py:98) */
    int max_cells;
    int log_rows;              /* rows of `log` per map (= num_iterations), 0 if log is NULL */
    mpp_ant_result *result;    /* [n_maps][n_total] */
    double *deposit;           /* [n_maps][n_total] Q/length per ant, 0 = deposits nothing (MAACO.py:307-308) */
    uint32_t *okbits;          /* [n_maps][ceil(n_total/32)] bit = ant deposits */
    mpp_maaco_state *state;    /* [n_maps] */
    int32_t *best_cells;       /* [n_maps][max_cells + 1] best path so far, decoded */
    double *log;               /* [n_maps][log_rows][4] = iter best len, iter best turns, overall len, overall turns; or NULL */
    unsigned long long *steps; /* [1] += ant steps taken; or NULL */
    const uint64_t *seeds;     /* [n_maps] Philox seed of each map's colony */
    const int32_t *latch;      /* NULL, or (sharded colony) != 0 once an exchange overflowed: every kernel is then a no-op */
} mpp_colony;

long long mpp_maaco_rank_words(int rows, int cols);
long long mpp_maaco_slab_words(int tile_rows, int cols, int n_ants);
long long mpp_maaco_touched_words(int tile_rows, int cols, int n_ants);

/* replaces MAACO._initialize_pheromones_maaco (MAACO.py:58-84), _precompute_dist_to_target
 * (:86-91) and the per-candidate heuristic eta'**beta (:197-210, :238) folded into two per-cell
 * tables E[cell][c], c = turn flag (interleaved: E01_dev[2*cell + c], 2*rows*cols doubles).  exp/pow
 * are evaluated on the host with libm (the same functions CPython/NumPy call) so the tables are
 * bit-identical to the reference.  The tables depend on (shape, start, target, parameters) only, so the maps of a
 * batch -- which must share start and target -- share ONE E01 / dist_t table (computed once), and tau0 of map k is
 * the shared free-cell table with map k's obstacles set to 1e-9 (a device kernel).  tau0_dev: [n_maps][tau_stride];
 * E01_dev: 2*rows*cols; dist_t_dev: rows*cols or NULL.  Synchronous. */
int mpp_maaco_tables(const mpp_map_batch *maps, const mpp_maaco_params *p, double *tau0_dev, long long tau_stride,
                     double *E01_dev, double *dist_t_dev, void *stream);

/* The tables of a batch whose maps have their own start and target (colony->E01_stride = 2*rows*cols):
 * mpp_maaco_e01_host: replaces the per-candidate heuristic eta'**beta (MAACO.py:197-210, :238) for n endpoint pairs
 *   (start[k], target[k]) of a rows x cols map: out [n][2*rows*cols], interleaved by turn flag, table k bit for bit
 *   what mpp_maaco_tables writes for a batch with those endpoints (the same host code, libm exp/pow).  Pure host code:
 *   touches no device, may run on any thread.  threads = 0: at most 16 (one below 65536 cells in all); the work is
 *   spread over maps and rows.  A cell outside 0..rows*cols-1 or n < 0 is an MPP_EINVAL.  Synchronous.
 * mpp_maaco_tau0_maps: replaces MAACO._initialize_pheromones_maaco (MAACO.py:58-84) for every map of the batch from
 *   that map's own start and target, obstacles at 1e-9 (:62-63): one kernel (grid.y = map) whose values are bit for bit
 *   mpp_maaco_tables' (integer squared distances, correctly rounded sqrt and division, no FMA).  tau0_dev:
 *   [n_maps][tau_stride].  Asynchronous on `stream`.  No dist_to_target table is produced.
 * mpp_maaco_e01_maps: mpp_maaco_e01_host on the device for every map of the batch from that map's own start and
 *   target: one thread per cell (grid.y = map), each writing its (E0, E1) pair as one 16-byte store.  exp / pow are
 *   mpp_exp / mpp_pow (csrc/mpp_libm.cuh), replicas of the x86-64 glibc 2.39 FMA-build functions, so the tables are
 *   bit for bit mpp_maaco_e01_host's where the host's libm is that build.  E01_dev: [n_maps][E01_stride] doubles,
 *   16-byte aligned, E01_stride even and >= 2*rows*cols.  A map without start or target is an MPP_EINVAL.
 *   Asynchronous on `stream`.
 * mpp_libm_exp_pow: out[2i] = mpp_exp(e[i]), out[2i+1] = mpp_pow(x[i], y[i]) for i < n, on the device (all pointers
 *   device memory), with the code mpp_maaco_e01_maps runs; what a caller compares with the host's libm before it
 *   trusts the device tables.  Asynchronous on `stream`. */
int mpp_maaco_e01_host(int rows, int cols, int n, const int32_t *start, const int32_t *target, const mpp_maaco_params *p,
                       double *out, int threads);
int mpp_maaco_tau0_maps(const mpp_map_batch *maps, const mpp_maaco_params *p, double *tau0_dev, long long tau_stride,
                        void *stream);
int mpp_maaco_e01_maps(const mpp_map_batch *maps, const mpp_maaco_params *p, double *E01_dev, long long E01_stride,
                       void *stream);
int mpp_libm_exp_pow(int n, const double *e, const double *x, const double *y, double *out, int device, void *stream);

/* The same two per-map tables for a batch whose maps also have their own colony parameters: params_dev is a DEVICE array
 * of n_maps mpp_maaco_params, map k's entry read by the blocks of grid row k.
 * mpp_maaco_tau0_maps_p: mpp_maaco_tau0_maps with C0_initial_pheromone of params_dev[k] for map k (MAACO.py:58-84);
 *   bit for bit what mpp_maaco_tables writes for that map alone with those parameters.
 * mpp_maaco_e01_maps_p: mpp_maaco_e01_maps with beta, a_turn_coef, wh_max, wh_min and k_h_adaptive of params_dev[k]
 *   (MAACO.py:197-210, :238); bit for bit mpp_maaco_e01_host's table of map k under its parameters where the host's
 *   libm is the build mpp_exp / mpp_pow reproduce.
 * A null params_dev or a map without start or target is an MPP_EINVAL.  Asynchronous on `stream`. */
int mpp_maaco_tau0_maps_p(const mpp_map_batch *maps, const mpp_maaco_params *params_dev, double *tau0_dev,
                          long long tau_stride, void *stream);
int mpp_maaco_e01_maps_p(const mpp_map_batch *maps, const mpp_maaco_params *params_dev, double *E01_dev,
                         long long E01_stride, void *stream);

/* replaces MAACO._calculate_adaptive_q0 (MAACO.py:212-226); pure host function */
double mpp_maaco_q0(int num_iterations, int iteration, double q0_initial);

/* ranks, per cell and previous-move context, the 8 moves by attractiveness tau**alpha * eta'**beta
 * (MAACO.py:235-239) into colony->rank.  Where every value is < 1e-10 the selection rules (:241-262) depend only on
 * that order and the tour kernel uses the ranking; elsewhere the entry says "evaluate".  Must be re-run after every
 * pheromone update.
 * alpha != 1: tau**alpha is CUDA's pow() (<= 2 ulp from glibc's, which is what NumPy calls at MAACO.py:238), so the
 * attractiveness values agree with the reference to ~4e-16 relative, NOT bit for bit: a discrete choice can differ
 * only where two candidate moves' attractiveness agree to that precision without being equal by symmetry.  alpha == 1
 * (the reference's default, x**1.0 == x) is exact. */
int mpp_maaco_rank(const mpp_map_batch *maps, const mpp_colony *colony, double alpha, void *stream);

/* replaces the ant loop MAACO.py:340-342 -> _construct_ant_solution_maaco (:278-302) with the
 * orientation filter + crossing-prohibition (:100-181) and pseudo-random-proportional selection
 * (:228-262), for ants [ant_offset, ant_offset + n_ants) of every map's colony (global ant id = RNG stream id).
 * Needs colony->rank of the CURRENT tau.  Writes slabs / touched (parity = iteration & 1) / moves of the n_ants local
 * ants and result[map][ant_offset + i].  ants_per_warp: 0 = chosen from the total load, or 1,2,4,..,32. */
int mpp_maaco_tours(const mpp_map_batch *maps, const mpp_colony *colony, int iteration, double q0, double alpha,
                    int n_ants, int ant_offset, int n_ants_total, int ants_per_warp, void *stream);

/* The same for a colony sharded over GPUs that can address each other's memory (NVLink peer memory): besides its local
 * buffers the kernel stores every visited-set slab straight into the receive buffers of the rank that updates that tile
 * row -- slabs_peers[g] = rank g's slabs_recv [tile_rows_per_rank x tile cols][n_ants_total][32], touched_peers[g]
 * its touched_recv (both parities) -- and every result into every rank's table result_peers[g][n_ants_total]; the three
 * arrays are HOST arrays of n_peers (<= 16) peer-mapped device pointers (they travel in the kernel's parameters).  After
 * one barrier across the ranks each of them runs mpp_maaco_best and mpp_maaco_pheromone (clear_slabs = 0) on what it
 * received: no pack / all-gather / replay step.  (The deposit MAACO.py:306-311 stays a sum over ALL ants in global
 * order on the rank that owns the cell.)  A single map only. */
int mpp_maaco_tours_p2p(const mpp_map_batch *maps, const mpp_colony *colony, int iteration, double q0, double alpha,
                        int n_ants, int ant_offset, int n_ants_total, int ants_per_warp,
                        uint32_t *const *slabs_peers, uint32_t *const *touched_peers,
                        mpp_ant_result *const *result_peers, int n_peers, int tile_rows_per_rank, void *stream);
/* the largest n_peers mpp_maaco_tours_p2p takes: a group of more ranks exchanges through mpp_maaco_xpack / _xunpack */
int mpp_maaco_max_peers(void);

/* replaces the order-dependent best tracking MAACO.py:343-358 for one iteration over all n_ants_total results of each
 * map (global ant order) and prepares deposit / okbits (:307-308).  Updates state and appends to log.  colony->moves
 * holds the tours of ants [moves_ant_offset, moves_ant_offset + moves_n_ants) (a sharded colony keeps only its own);
 * the new overall-best path is decoded into best_cells when the best ant lies in that range. */
int mpp_maaco_best(const mpp_map_batch *maps, const mpp_colony *colony, int moves_ant_offset, int moves_n_ants,
                   int n_ants_total, double Q, int iteration, void *stream);

/* replaces MAACO._update_pheromone_trails_maaco (MAACO.py:304-332) for the cells of tile rows
 * [tile_row0, tile_row0 + buf_tile_rows): evaporate, deposit in global ant order (bit-exact, atomics-free: one warp per
 * row of 32 cells walks the ants that have a slab for its tile), MMAS clip with tau_max from state->best_len,
 * obstacles <- 1e-9.  slabs_dev / touched_dev are laid out like colony->slabs / touched but cover buf_tile_rows tile rows
 * starting at tile_row0 and n_ants_total ants (single GPU: the colony's own buffers, tile_row0 = 0,
 * buf_tile_rows = TR; sharded: the receive buffers mpp_maaco_xunpack fills).  Clears the `touched` buffer of the next
 * pass, and (clear_slabs != 0) the slab words it read.  tau_peers_dev (optional, sharded colony over NVLink peer memory):
 * device array of n_peers pointers to every rank's pheromone field (this rank's included); the updated values are then
 * stored straight into all of them -- the all-gather of the tau slices fused into the update -- instead of colony->tau. */
int mpp_maaco_pheromone(const mpp_map_batch *maps, const mpp_colony *colony, uint32_t *slabs_dev, uint32_t *touched_dev,
                        int n_ants_total, int tile_row0, int buf_tile_rows, double rho, int iteration, int clear_slabs,
                        double *const *tau_peers_dev, int n_peers, void *stream);

/* one whole pass of a non-sharded colony: rank + tours + best + pheromone, enqueued on `stream` (asynchronous) */
int mpp_maaco_pass(const mpp_map_batch *maps, const mpp_colony *colony, const mpp_maaco_params *p, int iteration,
                   int n_ants, int ants_per_warp, void *stream);

/* mpp_maaco_pass with per-map colony parameters -- one iteration of MAACO.solve_path_planning's loop
 * (MAACO.py:336-359) for every map under ITS parameters, as if each map were solved alone with them.  params_dev: DEVICE
 * array of n_maps mpp_maaco_params (alpha, Q and rho are read here; num_iterations is not); q0_dev: DEVICE table
 * [num_iterations][n_maps] with q0_dev[(k-1) * n_maps + m] = mpp_maaco_q0(num_iterations, k, q0_initial of map m)
 * (MAACO.py:212-226), row iteration-1 is read.  The four kernels are per-map instantiations of mpp_maaco_pass's and
 * give map m the bits mpp_maaco_pass gives a one-map batch with map m's parameters (alpha != 1 included: both run CUDA's
 * pow for tau**alpha, see mpp_maaco_rank).  colony->E01 may be shared (E01_stride 0) when every map shares its endpoints
 * and table parameters, or per map (mpp_maaco_e01_maps_p).  A null params_dev / q0_dev, iteration < 1 or a map without
 * start or target is an MPP_EINVAL.  Asynchronous on `stream`. */
int mpp_maaco_pass_maps(const mpp_map_batch *maps, const mpp_colony *colony, const mpp_maaco_params *params_dev,
                        const double *q0_dev, int iteration, int n_ants, int ants_per_warp, void *stream);

/* mpp_maaco_pass_maps with a colony size and a pass count per map: map m is solved as if alone with
 * sizes_dev[m] = {num_ants, num_iterations} (DEVICE, [n_maps][2] int32).  n_ants is the colony's ant CAPACITY, the count
 * the buffers are laid out for (slabs, touched, moves, result, deposit and okbits strides); q0_dev is [max K][n_maps]
 * with column m = mpp_maaco_q0(K_m, k, q0_initial of map m) and must hold row iteration-1.  For map m:
 *   - its colony is n_m = num_ants clamped to [0, n_ants]: ants [0, n_m) construct tours, take part in the best scans
 *     and deposit; ants [n_m, n_ants) write no result, no slab, no `touched` bit and no step count, and get deposit 0.
 *     n_m = 0 constructs no tour and deposits nothing (tau still evaporates);
 *   - it takes part in pass `iteration` only if iteration <= num_iterations: past it (a negative count included) no
 *     kernel touches the map, so its tau, state, best path, log and results stay as they are.
 * sizes_dev = NULL is mpp_maaco_pass_maps (every map runs every pass with n_ants ants). */
int mpp_maaco_pass_maps_sized(const mpp_map_batch *maps, const mpp_colony *colony, const mpp_maaco_params *params_dev,
                              const double *q0_dev, const int32_t *sizes_dev, int iteration, int n_ants,
                              int ants_per_warp, void *stream);

/* the same pass with HOST buffers -- what a caller holding NumPy arrays binds: copies the pheromone field in
 * (tau_in_host: n_maps x rows*cols doubles, or NULL to keep the device field), runs the pass, copies out the updated
 * field, the per-ant results (n_maps x n_ants), the colony state(s) and the best path(s) so far
 * (n_maps x best_cells_capacity int32); any output pointer may be NULL.  SYNCHRONOUS: returns when the outputs are
 * valid.  replaces one iteration of MAACO.solve_path_planning's loop, MAACO.py:336-359. */
int mpp_maaco_pass_host(const mpp_map_batch *maps, const mpp_colony *colony, const mpp_maaco_params *p, int iteration,
                        int n_ants, int ants_per_warp, const double *tau_in_host, double *tau_out_host,
                        mpp_ant_result *result_out_host, mpp_maaco_state *state_out_host, int32_t *best_cells_out_host,
                        int best_cells_capacity, void *stream);

/* ---- sharded-colony exchange (no reference counterpart: the reference is single-process; these implement the
 * per-iteration exchange BASELINE's north star asks for, bit-exactly) ----------------------------------------
 * Rank g ships the results and the tours (1-byte move codes) of its n_local ants in ONE buffer per pass:
 *   [n_local x mpp_ant_result][int32 total code bytes + 12 pad bytes][codes: `capacity` bytes]
 * (mpp_maaco_xhdr_bytes(n_local) + capacity bytes; one all-gather moves it to every rank).
 * mpp_maaco_xpack   fills this rank's buffer from colony->result / moves (offsets_local_dev: n_local int32 scratch).
 *   With peer_xbuf_dev (device array of n_peers pointers to every rank's gathered buffer, NVLink peer memory) it writes
 *   slot `rank` of all of them directly instead -- the all-gather fused into the producer; the caller then only needs a
 *   barrier between the ranks.
 * mpp_maaco_xunpack on the gathered buffers (n_seg = ranks, seg_ants = ants per rank): copies all results into
 *   colony->result, computes per-ant code offsets (offsets_dev: n_seg*seg_ants int32), replays every ant's codes into
 *   the receive slabs / touched of tile rows [tile_row0, tile_row0 + buf_tile_rows) -- the input of
 *   mpp_maaco_pheromone (slabs_recv_dev must be zero on entry: the update clears what it read) -- and clears the
 *   parity-(iteration+1) half of the rank's own touched_local_dev.  If a segment's codes exceed `capacity` or a tour
 *   exceeds max_cells, *colony->latch is set to `iteration` (identically on every rank) and every later kernel is a
 *   no-op until the host clears it and repeats the pass with more room. */
long long mpp_maaco_xhdr_bytes(int n_local);
int mpp_maaco_xpack(const mpp_map_batch *maps, const mpp_colony *colony, int ant_offset, int n_local, int n_ants_total,
                    int32_t *offsets_local_dev, uint8_t *xbuf_local_dev, long long capacity,
                    uint8_t *const *peer_xbuf_dev, int n_peers, int rank, void *stream);
int mpp_maaco_xunpack(const mpp_map_batch *maps, const mpp_colony *colony, const uint8_t *xbuf_all_dev, long long capacity,
                      int n_seg, int seg_ants, int iteration, int32_t *offsets_dev, int tile_row0, int buf_tile_rows,
                      uint32_t *slabs_recv_dev, uint32_t *touched_recv_dev, uint32_t *touched_local_dev, void *stream);

/* ---- A* connectors, waypoint-chain fitness, path statistics (astar.py, MPA.py, helper.py, pso.py, ga_solver.py) ---- */
typedef struct {
    double turn_penalty_factor, safety_penalty_factor, min_safe_distance, diagonal_obstacle_penalty_value;
    int restrict_policy;  /* restrict_diagonal_near_obstacle_policy: connector bans corner cutting; stats charge it */
    int allow_diagonal;   /* allow_diagonal_moves */
    int mode;             /* 0 = helper.calculate_path_stats, 1 = MPA._calculate_path_stats (safety hard-wired 0.0) */
} mpp_policy;

/* replaces calculate_path_safety_penalty's O(len x n_obstacles) scan (helper.py:67-80) by a per-cell class
 * table (u16: min squared distance to an obstacle within floor(msd)) + a LUT of (msd - d)**2 per class, evaluated
 * with libm on the host.  0 <= msd <= 180 (u16 classes).  One launch (grid.y = map) builds [n_maps][rows*cols] classes;
 * one LUT is shared by all maps (it depends on msd only).  Cached in the batch for one msd at a time; called implicitly
 * by every entry point that computes statistics in mode 0. */
int mpp_map_batch_safety_table(mpp_map_batch *maps, double min_safe_distance, void *stream);

/* replaces helper.calculate_path_stats (helper.py:98-113; count_turns :58-65, safety :67-80, diagonal
 * penalty :82-96) and MPA._calculate_path_stats (MPA.py:215-229) for n_paths paths, one warp each; path i lies on map
 * map_dev[i].  length uses CPython 3.12's Neumaier-compensated sum().  stats_dev: n_paths x 5 doubles =
 * (length, turns, safety_penalty, diag_penalty, fitness); an empty path, or one whose map index lies outside the batch
 * -> (inf, 0, 0, 0, inf). */
int mpp_path_stats(mpp_map_batch *maps, const int32_t *map_dev, const int32_t *cells_dev, int max_cells,
                   const int32_t *n_cells_dev, int n_paths, const mpp_policy *policy, double *stats_dev, void *stream);

/* search slots (one lane group each) of a batch that are resident at once; the scratch of the search entry points is
 * 256 + n_slots * mpp_astar_slot_bytes(rows, cols, heap_cap) bytes for n_slots concurrent searches with a heap of
 * heap_cap entries each, zero-filled once before its first use (search stamps live in it). */
int mpp_map_batch_max_slots(const mpp_map_batch *maps);

/* replaces n independent calls of AStarSolver.solve (variant 0, astar.py:33-101, with get_valid_neighbors
 * helper.py:18-53), MPA._a_star (variant 1, MPA.py:106-151) or DijkstraSolver.solve (variant 2,
 * dijkstra.py:32-97 = variant 0 with a zero heuristic), on a batch of same-shape maps in one launch -- with map
 * indices, also one AStarSolver(grid).solve() / DijkstraSolver(grid).solve() per map of a sweep over independent maps.
 * Query i runs on map map_dev[i] (any number of queries per map, each with its own endpoints and avoid set); a query
 * whose map index or endpoint lies outside the batch / map gets n_cells = 0 without a search.  avoid_bits_dev:
 * optional n x ceil(rows*cols/32) bitmaps (nodes_to_avoid).  cells_dev: n x max_cells; n_cells_dev[i] = path length
 * (0 = no path / invalid endpoint, -1 = heap_cap overflow, > max_cells = truncated); g_dev[i] = g of the popped
 * target (nullable).  counters_dev: optional [4] = (node expansions, successful relaxations, ring-bucket pushes,
 * overflow-heap pushes), accumulated.  stats_policy (nullable): the lane group computes the statistics of its own path
 * right after the search into stats_dev (n x 5, as mpp_path_stats; mode 0 uses that map's safety table,
 * mpp_map_batch_safety_table); a query with n_cells <= 0 or > max_cells gets the empty path's (inf, 0, 0, 0, inf).
 * order_dev: optional permutation of 0..n-1 = the order in which free slots take the queries (start the long ones
 * first); results stay indexed by query.  n_slots <= mpp_map_batch_max_slots is useful.  A one-map batch whose
 * occupancy fits is staged in shared memory by every block; larger maps and batches of several maps read it through
 * L2. */
int mpp_astar_batch_maps(mpp_map_batch *maps, int variant, const int32_t *map_dev, const int32_t *src_dev,
                         const int32_t *dst_dev, const uint32_t *avoid_bits_dev, int n, int allow_diagonal,
                         int restrict_corner, const mpp_policy *stats_policy, int32_t *cells_dev, int max_cells,
                         int32_t *n_cells_dev, double *g_dev, double *stats_dev, void *scratch_dev, size_t scratch_bytes,
                         int n_slots, int heap_cap, unsigned long long *counters_dev, const int32_t *order_dev,
                         void *stream);

/* ---- exact Dijkstra distance fields (dijkstra.py) -----------------------------------------------------------------
 * replaces DijkstraSolver.solve's search (dijkstra.py:32-97, with get_valid_neighbors helper.py:18-53) when one source
 * serves many targets, or a whole map's costs are wanted: ONE field per map gives every target's popped g and path.
 * mpp_dijkstra_fields: for every map k of the batch (a single map: a batch of one), the complete field from cell
 *   src_dev[k]: g_dev [n_maps][rows*cols] = the g with which dijkstra.py pops each cell (+inf: obstacle or unreachable),
 *   parent_dev [n_maps][rows*cols] = the move parent -> cell in the move order of helper.py:30-36 ((0,1), (0,-1), (1,0),
 *   (-1,0), (1,1), (1,-1), (-1,1), (-1,-1)), 0xFF = none (source, obstacle, unreachable).  Both are bit for bit what the
 *   reference's search computes for that cell as its target: g*(cell) is the least fixed point of the relaxations
 *   (fp64 rounding is monotone and every step weighs >= 1), the parent the first strict improvement in (g, r, c) pop
 *   order.  A source outside the map or on an obstacle gives an all-inf field.  scratch: mpp_dijkstra_field_scratch_bytes
 *   bytes, no initialisation needed.  One thread-block cluster per map (up to 16 CTAs when the batch has few maps).
 * mpp_dijkstra_field_paths: query i reads the path from the source of map map_dev[i]'s field to cell dst_dev[i]
 *   (dijkstra.py:64-70): cells_dev n x max_cells, n_cells_dev[i] = path length (0 = unreachable / obstacle / endpoint or
 *   map index outside the batch, > max_cells = truncated), g_out_dev[i] = g*(dst) (+inf without a path; nullable), and
 *   with stats_policy the statistics into stats_dev as mpp_astar_batch_maps computes them.  A target equal to the source
 *   gives [src] with g = 0.  One lane group (warp) per query. */
size_t mpp_dijkstra_field_scratch_bytes(const mpp_map_batch *maps);
int mpp_dijkstra_fields(const mpp_map_batch *maps, const int32_t *src_dev, int allow_diagonal, int restrict_corner,
                        double *g_dev, uint8_t *parent_dev, void *scratch_dev, size_t scratch_bytes, void *stream);
int mpp_dijkstra_field_paths(mpp_map_batch *maps, const double *g_dev, const uint8_t *parent_dev, const int32_t *map_dev,
                             const int32_t *dst_dev, int n, const mpp_policy *stats_policy, int32_t *cells_dev,
                             int max_cells, int32_t *n_cells_dev, double *g_out_dev, double *stats_dev, void *stream);

/* replaces PSOSolver._reconstruct_path_from_position (pso.py:56-94, after rounding/clamping) /
 * GASolver._reconstruct_path_from_chromosome (ga_solver.py:58-93) followed by
 * BasePathfinder._calculate_stats_for_path (helper.py:138-147) for whole populations, on a batch of same-shape maps in
 * one launch: one lane group (a warp) per individual runs its W+1 connector searches with the growing avoid set and the
 * statistics of the joined path.  Individual i runs on map map_dev[i] from that map's start, through its waypoints
 * (waypoints_dev: N x W cells), to that map's target; mode 0 uses that map's safety table (mpp_map_batch_safety_table).
 * An individual whose map index lies outside the batch (or whose map has no start / target) gets n_cells = 0 without a
 * search.  visited_dev: n_slots x ceil(rows*cols/32) words of scratch (one bitmap per search slot).  Scratch as
 * mpp_astar_batch_maps.  n_cells_dev[i]: 0 = invalid individual ([]), -1 = heap overflow, > max_cells = truncated.
 * order_dev: optional permutation of 0..N-1 = the order in which free search slots take individuals (the evaluation
 * lasts as long as its longest chain of searches: start the long ones first); results stay indexed by individual.
 * Occupancy staging as mpp_astar_batch_maps. */
int mpp_waypoint_fitness_maps(mpp_map_batch *maps, const int32_t *map_dev, const int32_t *waypoints_dev,
                              int n_individuals, int n_waypoints, const mpp_policy *policy, int32_t *cells_dev,
                              int max_cells, int32_t *n_cells_dev, double *stats_dev, uint32_t *visited_dev,
                              void *scratch_dev, size_t scratch_bytes, int n_slots, int heap_cap,
                              unsigned long long *counters_dev, const int32_t *order_dev, void *stream);

/* ---- per-map parameters of the population planners (a parameter sweep as one batch) --------------------------------
 * One entry per map of a batch, kept by the caller in a DEVICE array params_dev[n_maps]; map m's entry is read by the
 * blocks (or lane groups) that work on map m.  Each planner reads its own fields and the three statistics weights:
 *   PSO: w, c1, c2 (pso.py:185-190); GA: crossover_rate, mutation_rate, tournament_size (ga_solver.py:136-160);
 *   MPA: P_const, FADs_rate, levy_sigma (MPA.py:251-253, computed by the caller), levy_beta (MPA.py:10-18);
 *   the statistics: turn_penalty_factor, safety_penalty_factor, diagonal_obstacle_penalty_value (helper.py:98-113,
 *   MPA.py:215-229) in place of the mpp_policy fields of those names.
 * What changes the search or the safety tables -- min_safe_distance, allow_diagonal, restrict_policy, mode -- stays in
 * the mpp_policy argument and is common to the batch. */
typedef struct {
    double w, c1, c2;
    double crossover_rate, mutation_rate;
    int tournament_size;
    double P_const, FADs_rate, levy_sigma, levy_beta;
    double turn_penalty_factor, safety_penalty_factor, diagonal_obstacle_penalty_value;
} mpp_pop_params;

/* mpp_waypoint_fitness_maps / mpp_path_stats with the statistics weights of params_dev[m] for an individual / path on
 * map m (an individual or path outside the batch gets the empty path's statistics, as there); the searches are those of
 * the functions without _p.  For map m the results are bit for bit what the function without _p gives with a policy
 * carrying params_dev[m]'s weights.  A null params_dev is an MPP_EINVAL. */
int mpp_waypoint_fitness_maps_p(mpp_map_batch *maps, const int32_t *map_dev, const int32_t *waypoints_dev,
                                int n_individuals, int n_waypoints, const mpp_policy *policy,
                                const mpp_pop_params *params_dev, int32_t *cells_dev, int max_cells,
                                int32_t *n_cells_dev, double *stats_dev, uint32_t *visited_dev, void *scratch_dev,
                                size_t scratch_bytes, int n_slots, int heap_cap, unsigned long long *counters_dev,
                                const int32_t *order_dev, void *stream);
int mpp_path_stats_p(mpp_map_batch *maps, const int32_t *map_dev, const int32_t *cells_dev, int max_cells,
                     const int32_t *n_cells_dev, int n_paths, const mpp_policy *policy,
                     const mpp_pop_params *params_dev, double *stats_dev, void *stream);

/* ---- MPA (MPA.py) ------------------------------------------------------------------------------- */

/* MPA over a batch of independent same-shape maps (BASELINE config 5; a single map is a batch of one), one launch per
 * iteration for every map.  Population buffers are [n_maps][n_predators][...] (cells: max_cells int32 per predator;
 * stats: 5 doubles).
 * mpp_mpa_init_batch: MPA._initialize_population_with_safety (MPA.py:231-245) -- ONE private-A* search start -> target
 *   per map (the reference runs N identical ones); writes row 0 of every map (path, n_cells, stats); the caller
 *   replicates it.  scratch: 256 + n_maps * mpp_astar_slot_bytes(rows, cols, heap_cap).
 * mpp_mpa_iteration_batch: replaces one iteration of MPA.solve_path_planning for the whole population (MPA.py:339-410)
 *   of every map: the phase loop (:340-377: start index + gate draw, Levy :250-264 / Brownian :266-282 target,
 *   _reconstruct_path_segment :284-318 with the private A* :106-151 and stats :215-229), the marine-memory step
 *   (:380-384) and the FADs step (:387-410).  The old population must be sorted by fitness (row 0 = elite, :333-334)
 *   -- or order_dev [n_maps][n_predators] is the stable argsort of its fitness column (the sorts of MPA.py:333,412 as an
 *   index, no path is moved): predator i reads row order[i], the elite is row order[0] (null: the identity).  The next
 *   population is written unsorted to row i of the out buffers.  phase = 1/2/3 (:339,:348,:365), CF as computed at
 *   :336, levy_sigma as at :251-253.  Only predators [pred_begin, pred_end) of every map are processed (a rank's shard
 *   of the population; their rows of out_* are written).  seeds_dev: one Philox seed per map; streams (seed, MPA_PHASE,
 *   iteration, i) and (seed, MPA_FADS, iteration, i).  tmp_cells_dev: n_maps * warps_per_map x max_cells, avoid_dev:
 *   n_maps * warps_per_map x ceil(rows*cols/32) words of scratch; queue_dev: n_maps uint32 scratch; scratch:
 *   256 + n_maps * warps_per_map slots.  status_dev[0] (zero it first): 1 = heap overflow, 2 = a path exceeded
 *   max_cells (repeat with larger buffers).  The occupancy is staged in shared memory when it fits. */
int mpp_mpa_init_batch(const mpp_map_batch *maps, const mpp_policy *policy, int n_predators, int max_cells,
                       int32_t *cells_dev, int32_t *n_cells_dev, double *stats_dev, void *scratch_dev,
                       size_t scratch_bytes, int heap_cap, int32_t *status_dev, unsigned long long *counters_dev,
                       void *stream);
int mpp_mpa_iteration_batch(const mpp_map_batch *maps, const mpp_policy *policy, int n_predators, int pred_begin,
                            int pred_end, int iteration, int phase,
                            double P_const, double CF, double FADs_rate, double levy_sigma, double levy_beta,
                            const uint64_t *seeds_dev, const int32_t *order_dev, const int32_t *cells_dev,
                            const int32_t *n_cells_dev, const double *stats_dev, int max_cells, int32_t *out_cells_dev,
                            int32_t *out_n_dev, double *out_stats_dev, int32_t *tmp_cells_dev, uint32_t *avoid_dev,
                            void *scratch_dev, size_t scratch_bytes, int warps_per_map, int heap_cap, uint32_t *queue_dev,
                            int32_t *status_dev, unsigned long long *counters_dev, void *stream);
/* The same two steps for a batch whose maps have their own MPA parameters (mpp_pop_params above): map m reads P_const,
 * FADs_rate, levy_sigma and levy_beta (1 / levy_beta is an IEEE division, as mpp_mpa_iteration_batch computes it) and
 * the three statistics weights from params_dev[m] in place of the scalars and the policy's weights; map m's results are
 * bit for bit those of the functions without _p given map m's values.  A null params_dev is an MPP_EINVAL. */
int mpp_mpa_init_batch_p(const mpp_map_batch *maps, const mpp_policy *policy, const mpp_pop_params *params_dev,
                         int n_predators, int max_cells, int32_t *cells_dev, int32_t *n_cells_dev, double *stats_dev,
                         void *scratch_dev, size_t scratch_bytes, int heap_cap, int32_t *status_dev,
                         unsigned long long *counters_dev, void *stream);
int mpp_mpa_iteration_batch_p(const mpp_map_batch *maps, const mpp_policy *policy, int n_predators, int pred_begin,
                              int pred_end, int iteration, int phase, const mpp_pop_params *params_dev, double CF,
                              const uint64_t *seeds_dev, const int32_t *order_dev, const int32_t *cells_dev,
                              const int32_t *n_cells_dev, const double *stats_dev, int max_cells, int32_t *out_cells_dev,
                              int32_t *out_n_dev, double *out_stats_dev, int32_t *tmp_cells_dev, uint32_t *avoid_dev,
                              void *scratch_dev, size_t scratch_bytes, int warps_per_map, int heap_cap,
                              uint32_t *queue_dev, int32_t *status_dev, unsigned long long *counters_dev, void *stream);
/* bytes of one search slot's scratch for a rows x cols map */
size_t mpp_astar_slot_bytes(int rows, int cols, int heap_cap);

/* ---- PSO / GA population updates (pso.py, ga_solver.py) ------------------------------------------------------------
 * One launch per step for every map of a batch (grid.y = map): map m's arrays are row m of [n_maps][...] buffers, and
 * it draws from the streams of seeds_dev[m] -- exactly what a per-map solver with rng_seed = seeds[m] draws (a single
 * solver passes a one-map batch and one seed).  With several maps they replace a Python loop
 * `for grid in grids: PSOSolver(grid, ...).solve()` / `GASolver(grid, ...).solve()`.
 * mpp_pso_init_batch: replaces the attempt generation of PSOSolver._initialize_particles (pso.py:97-105: W uniform
 *   waypoints + W x 2 uniform velocities per attempt, :50-51, the rounded, clamped cells :61, :69-70) for attempts
 *   [off[m], off[m] + n_attempts) of every map with attempt_offset_dev[m] >= 0 (a negative offset: the map is done, its
 *   rows are not written).  pos / vel: [n_maps][n_attempts][W][2], waypoint cells [n_maps][n_attempts][W].  Stream
 *   (seed, PSO_INIT, 0, attempt).  The accept / pad bookkeeping (pso.py:107-160) stays with the caller.
 * mpp_ga_init_batch: replaces GASolver._create_chromosome (ga_solver.py:48-56: integer genes redrawn until the cell is
 *   free) for the attempts of _initialize_population (:95-104) -- the same for chromosomes [n_maps][n_attempts][W].
 *   Stream (seed, GA_INIT, 0, attempt).
 * mpp_pso_update_batch: replaces the velocity/position update of the particle loop (pso.py:183-206) for particles
 *   [start_dev[m], n_particles) of map m (start = n_particles: the map is idle; the particles below start are not
 *   touched; a suffix is re-run when an earlier particle improved gbest -- the reference's loop is asynchronous,
 *   pso.py:222-229).  pos / vel / pbest: [n_maps][n_particles][W][2] doubles (row, col), gbest [n_maps][W][2].  Exactly
 *   4W uniforms per particle, stream (seed, PSO_UPDATE, iteration, particle).  Also writes the integer waypoints
 *   pso.py:61,69-70 (round-half-even, clamped) as cells into waypoint cells [n_maps][n_particles][W].
 * mpp_ga_select_batch: replaces GASolver._selection (ga_solver.py:136-142) over fitness [n_maps][n] (population,
 *   i.e. sorted, order) -> parents [n_maps][n] population indices: n tournaments of min(tournament_size, n)
 *   individuals drawn with CPython's random.sample algorithm (randbelow(n) = floor(u*n)); winner = first minimum in
 *   sample order.  Stream (seed, GA_SELECT, generation, tournament).
 * mpp_ga_breed_batch: replaces the breeding loop ga_solver.py:186-194 (_crossover :144-152, _mutate :154-160,
 *   _generate_random_waypoint :48-53) over chromosomes / children [n_maps][n][W] in population order: pair
 *   p = (parents[2p % n], parents[(2p+1) % n]) -> children 2p, 2p+1; mutated genes are free cells of the map's own
 *   grid.  Stream (seed, GA_BREED, generation, pair). */
int mpp_pso_init_batch(const mpp_map_batch *maps, int n_attempts, const int32_t *attempt_offset_dev, int n_waypoints,
                       double max_vel, const uint64_t *seeds_dev, double *pos_dev, double *vel_dev,
                       int32_t *waypoint_cells_dev, void *stream);
int mpp_ga_init_batch(const mpp_map_batch *maps, int n_attempts, const int32_t *attempt_offset_dev, int n_waypoints,
                      const uint64_t *seeds_dev, int32_t *chrom_dev, void *stream);
int mpp_pso_update_batch(const mpp_map_batch *maps, double *pos_dev, double *vel_dev, const double *pbest_pos_dev,
                         const double *gbest_pos_dev, int n_particles, const int32_t *start_dev, int n_waypoints,
                         double w, double c1, double c2, double max_vel, const uint64_t *seeds_dev, int iteration,
                         int32_t *waypoint_cells_dev, void *stream);
int mpp_ga_select_batch(const mpp_map_batch *maps, const double *fitness_dev, int n, int tournament_size,
                        const uint64_t *seeds_dev, int generation, int32_t *parents_dev, void *stream);
int mpp_ga_breed_batch(const mpp_map_batch *maps, const int32_t *chrom_dev, const int32_t *parents_dev, int n,
                       int n_waypoints, double crossover_rate, double mutation_rate, const uint64_t *seeds_dev,
                       int generation, int32_t *children_dev, void *stream);

/* The three update steps with per-map parameters: map m reads w, c1, c2 / tournament_size / crossover_rate,
 * mutation_rate from params_dev[m] (mpp_pop_params) in place of the scalars; everything else as above, and map m's
 * results are bit for bit those of the functions without _p given map m's values.  A map whose
 * k = min(tournament_size, n) the selection cannot take (k outside 1..16, or k > 5 with n <= 85: the scalar function
 * refuses such a launch) gets parents -1 in every slot; the breeding reads a parent index outside 0..n-1 as 0.  Neither
 * kernel reads or writes outside its buffers for any parameter value.  A null params_dev is an MPP_EINVAL. */
int mpp_pso_update_batch_p(const mpp_map_batch *maps, double *pos_dev, double *vel_dev, const double *pbest_pos_dev,
                           const double *gbest_pos_dev, int n_particles, const int32_t *start_dev, int n_waypoints,
                           const mpp_pop_params *params_dev, double max_vel, const uint64_t *seeds_dev, int iteration,
                           int32_t *waypoint_cells_dev, void *stream);
int mpp_ga_select_batch_p(const mpp_map_batch *maps, const double *fitness_dev, int n, const mpp_pop_params *params_dev,
                          const uint64_t *seeds_dev, int generation, int32_t *parents_dev, void *stream);
int mpp_ga_breed_batch_p(const mpp_map_batch *maps, const int32_t *chrom_dev, const int32_t *parents_dev, int n,
                         int n_waypoints, const mpp_pop_params *params_dev, const uint64_t *seeds_dev, int generation,
                         int32_t *children_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MPP_H_ */
