// mpp_pop.cu -- fused elementwise population updates: PSO velocity/position (pso.py:183-206),
// GA tournament selection / crossover / mutation (ga_solver.py:136-160).  One thread per
// (particle, waypoint) / tournament / parent pair; every uniform comes from the Philox stream of the
// RNG contract, so any rank can regenerate any individual's draws.
// Every kernel runs over a batch of maps with grid.y = map: map m's arrays are row m of [n_maps][...] buffers and
// its seed is seeds[m] (the same streams as a single-map solver with that seed); a single map is a batch of one.
#include "mpp_common.cuh"

#define MPP_POP_MAX_MAPS 65535                                 // grid.y


// ---------------------------------------------------------------------------------------------
// K8: PSO update.  v = ((w*v) + ((c1*r1)*(pbest-x))) + ((c2*r2)*(gbest-x)); clip; x = clip(x+v).
// Draw order per particle (pso.py:185-190): for each waypoint: r1,r2 (row) then r1',r2' (col)
// => draws 4*dim+{0,1,2,3} of stream (seed, PSO_UPDATE, iteration, particle).
// Also emits the integer waypoint pso.py:61,69-70: int(round(x)) (half-even) clamped to the grid.
// ---------------------------------------------------------------------------------------------
// Particles [start[m], n) of map m (the stream index is the particle index).
__global__ void mpp_pso_update_kernel(double *__restrict__ pos, double *__restrict__ vel,
                                      const double *__restrict__ pbest, const double *__restrict__ gbest, int n, int W,
                                      const int32_t *__restrict__ start, double w, double c1, double c2, double max_vel,
                                      int R, int C, const uint64_t *__restrict__ seeds, uint32_t iteration,
                                      int32_t *__restrict__ wp_cells) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * W) return;
    const int p = t / W, dim = t % W;
    if (p < start[blockIdx.y]) return;
    const uint64_t sd = seeds[blockIdx.y];
    const uint32_t k0 = (uint32_t)sd, k1 = (uint32_t)(sd >> 32);
    const size_t row = (size_t)blockIdx.y * n * W;             // map m's particles
    pos += 2 * row; vel += 2 * row; pbest += 2 * row; wp_cells += row;
    gbest += (size_t)blockIdx.y * W * 2;
    const mpp_u4 a = mpp_philox(2u * dim, (uint32_t)p, iteration, MPP_CLS_PSO_UPDATE, k0, k1);
    const mpp_u4 b = mpp_philox(2u * dim + 1u, (uint32_t)p, iteration, MPP_CLS_PSO_UPDATE, k0, k1);
    const double r1 = mpp_u53(a.x, a.y), r2 = mpp_u53(a.z, a.w), r3 = mpp_u53(b.x, b.y), r4 = mpp_u53(b.z, b.w);
    const size_t i = ((size_t)p * W + dim) * 2;
    const double xr = pos[i], xc = pos[i + 1];
    double vr = w * vel[i] + (c1 * r1) * (pbest[i] - xr) + (c2 * r2) * (gbest[2 * dim] - xr);          // :185-187
    double vc = w * vel[i + 1] + (c1 * r3) * (pbest[i + 1] - xc) + (c2 * r4) * (gbest[2 * dim + 1] - xc);  // :188-190
    vr = fmin(fmax(vr, -max_vel), max_vel);                                                           // :192-193
    vc = fmin(fmax(vc, -max_vel), max_vel);
    const double nr = fmin(fmax(xr + vr, 0.0), (double)(R - 1));                                      // :197-202
    const double nc = fmin(fmax(xc + vc, 0.0), (double)(C - 1));
    vel[i] = vr; vel[i + 1] = vc;
    pos[i] = nr; pos[i + 1] = nc;
    int ir = (int)rint(nr), ic = (int)rint(nc);                                                       // :61 round-half-even
    ir = max(0, min(R - 1, ir)); ic = max(0, min(C - 1, ic));                                         // :69-70
    wp_cells[(size_t)p * W + dim] = ir * C + ic;
}

extern "C" int mpp_pso_update_batch(const mpp_map_batch *maps, double *pos_dev, double *vel_dev,
                                    const double *pbest_pos_dev, const double *gbest_pos_dev, int n_particles,
                                    const int32_t *start_dev, int n_waypoints, double w, double c1, double c2,
                                    double max_vel, const uint64_t *seeds_dev, int iteration,
                                    int32_t *waypoint_cells_dev, void *stream) {
    MPP_REQUIRE(maps && pos_dev && vel_dev && pbest_pos_dev && gbest_pos_dev && start_dev && seeds_dev &&
                waypoint_cells_dev, "mpp_pso_update_batch: null argument");
    MPP_REQUIRE(n_particles > 0 && n_waypoints > 0 && maps->n_maps <= MPP_POP_MAX_MAPS, "mpp_pso_update_batch: bad sizes");
    MPP_CUDA(cudaSetDevice(maps->device));
    const int total = n_particles * n_waypoints;
    mpp_pso_update_kernel<<<dim3((total + 255) / 256, maps->n_maps), 256, 0, (cudaStream_t)stream>>>(
        pos_dev, vel_dev, pbest_pos_dev, gbest_pos_dev, n_particles, n_waypoints, start_dev, w, c1, c2, max_vel,
        maps->rows, maps->cols, seeds_dev, (uint32_t)iteration, waypoint_cells_dev);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

// ---------------------------------------------------------------------------------------------
// K9a: GA tournament selection (ga_solver.py:136-142).  random.sample(population, k) is CPython's
// algorithm with randbelow(n) = floor(u*n): pool variant for n <= setsize, set-rejection otherwise.
// winner = first minimum fitness in sample order.  Stream (seed, GA_SELECT, generation, tournament).
// ---------------------------------------------------------------------------------------------
#define MPP_GA_MAX_K 16
__global__ void mpp_ga_select_kernel(const double *__restrict__ fitness, int n, int k, const uint64_t *__restrict__ seeds,
                                     uint32_t generation, int32_t *__restrict__ parents) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    fitness += (size_t)blockIdx.y * n;
    parents += (size_t)blockIdx.y * n;
    mpp_stream_rng rng;
    rng.init(seeds[blockIdx.y], MPP_CLS_GA_SELECT, generation, (uint32_t)t);
    int setsize = 21;
    if (k > 5) {  // setsize += 4 ** ceil(log(k*3, 4))
        int e = 0, v = 1;
        while (v < k * 3) { v *= 4; ++e; }
        setsize += v;
    }
    int sel[MPP_GA_MAX_K];
    if (n <= setsize) {
        int pool[21 + 64];
        for (int i = 0; i < n; ++i) pool[i] = i;
        for (int i = 0; i < k; ++i) {
            const int j = rng.below(n - i);
            sel[i] = pool[j];
            pool[j] = pool[n - i - 1];
        }
    } else {
        for (int i = 0; i < k; ++i) {
            int j;
            bool dup;
            do {
                j = rng.below(n);
                dup = false;
                for (int q = 0; q < i; ++q) dup |= (sel[q] == j);
            } while (dup);
            sel[i] = j;
        }
    }
    int best = sel[0];
    double bf = fitness[best];
    for (int i = 1; i < k; ++i) {
        const double f = fitness[sel[i]];
        if (f < bf) { bf = f; best = sel[i]; }
    }
    parents[t] = best;
}

extern "C" int mpp_ga_select_batch(const mpp_map_batch *maps, const double *fitness_dev, int n, int tournament_size,
                                   const uint64_t *seeds_dev, int generation, int32_t *parents_dev, void *stream) {
    MPP_REQUIRE(maps && seeds_dev && fitness_dev && parents_dev && n > 0 && maps->n_maps <= MPP_POP_MAX_MAPS,
                "mpp_ga_select_batch: bad argument");
    int k = tournament_size < n ? tournament_size : n;  // min(tournament_size, len(population))
    MPP_REQUIRE(k >= 1 && k <= MPP_GA_MAX_K, "mpp_ga_select_batch: tournament size %d unsupported (1..%d)", k, MPP_GA_MAX_K);
    MPP_REQUIRE(k <= 5 || n > 21 + 64, "mpp_ga_select_batch: tiny population with large tournament unsupported");
    MPP_CUDA(cudaSetDevice(maps->device));
    mpp_ga_select_kernel<<<dim3((n + 127) / 128, maps->n_maps), 128, 0, (cudaStream_t)stream>>>(
        fitness_dev, n, k, seeds_dev, (uint32_t)generation, parents_dev);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

// ---------------------------------------------------------------------------------------------
// K9b: GA crossover + mutation (ga_solver.py:144-160, loop :186-194).  Thread per parent pair
// `pair` (parents[2*pair % n], parents[(2*pair+1) % n]) -> children slots 2*pair, 2*pair+1.
// Stream (seed, GA_BREED, generation, pair): crossover draw(s), then mutation of child 1, child 2.
// ---------------------------------------------------------------------------------------------
#define MPP_GA_MAX_W 64
__device__ __forceinline__ int ga_random_free_cell(mpp_stream_rng &rng, const uint32_t *occ, int pitch, int R, int C) {
    for (;;) {                                                         // ga_solver.py:48-53
        const int r = rng.below(R);
        const int c = rng.below(C);
        const int pb = c + 1;
        if (!((occ[(r + 1) * pitch + (pb >> 5)] >> (pb & 31)) & 1u)) return r * C + c;
    }
}

__global__ void mpp_ga_breed_kernel(const uint32_t *__restrict__ occ, int occ_words, int pitch, int R, int C,
                                    const int32_t *__restrict__ chrom, const int32_t *__restrict__ parents, int n, int W,
                                    double cx_rate, double mut_rate, const uint64_t *__restrict__ seeds,
                                    uint32_t generation, int32_t *__restrict__ children) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    const int n_pairs = (n + 1) / 2;
    if (pair >= n_pairs) return;
    occ += (size_t)blockIdx.y * occ_words;                     // mutated genes are free cells of the map's own grid
    chrom += (size_t)blockIdx.y * n * W;
    parents += (size_t)blockIdx.y * n;
    children += (size_t)blockIdx.y * n * W;
    mpp_stream_rng rng;
    rng.init(seeds[blockIdx.y], MPP_CLS_GA_BREED, generation, (uint32_t)pair);
    const int32_t *p1 = chrom + (size_t)parents[(2 * pair) % n] * W;
    const int32_t *p2 = chrom + (size_t)parents[(2 * pair + 1) % n] * W;
    int32_t c1[MPP_GA_MAX_W], c2[MPP_GA_MAX_W];
    int point = 0;
    if (rng.draw() < cx_rate && W > 0) {                               // :145
        point = (W > 1) ? 1 + rng.below(W - 1) : 0;                    // randint(1, W-1) :147
    }
    for (int i = 0; i < W; ++i) {                                      // :149-152
        const bool swap = point > 0 && i >= point;
        c1[i] = swap ? p2[i] : p1[i];
        c2[i] = swap ? p1[i] : p2[i];
    }
    for (int i = 0; i < W; ++i)                                        // _mutate(c1) :154-160
        if (rng.draw() < mut_rate) c1[i] = ga_random_free_cell(rng, occ, pitch, R, C);
    for (int i = 0; i < W; ++i)                                        // _mutate(c2)
        if (rng.draw() < mut_rate) c2[i] = ga_random_free_cell(rng, occ, pitch, R, C);
    for (int i = 0; i < W; ++i) children[(size_t)(2 * pair) * W + i] = c1[i];
    if (2 * pair + 1 < n)
        for (int i = 0; i < W; ++i) children[(size_t)(2 * pair + 1) * W + i] = c2[i];
}

extern "C" int mpp_ga_breed_batch(const mpp_map_batch *maps, const int32_t *chrom_dev, const int32_t *parents_dev, int n,
                                  int n_waypoints, double crossover_rate, double mutation_rate, const uint64_t *seeds_dev,
                                  int generation, int32_t *children_dev, void *stream) {
    MPP_REQUIRE(maps && chrom_dev && parents_dev && seeds_dev && children_dev && n > 0 && maps->n_maps <= MPP_POP_MAX_MAPS,
                "mpp_ga_breed_batch: bad argument");
    MPP_REQUIRE(n_waypoints >= 1 && n_waypoints <= MPP_GA_MAX_W, "mpp_ga_breed_batch: %d waypoints unsupported (1..%d)",
                n_waypoints, MPP_GA_MAX_W);
    for (int k = 0; k < maps->n_maps; ++k)                             // the start cell is free: mutation terminates
        MPP_REQUIRE(maps->meta_host[k].start >= 0, "mpp_ga_breed_batch: map %d has no start", k);
    MPP_CUDA(cudaSetDevice(maps->device));
    const int n_pairs = (n + 1) / 2;
    mpp_ga_breed_kernel<<<dim3((n_pairs + 127) / 128, maps->n_maps), 128, 0, (cudaStream_t)stream>>>(
        maps->occ_dev, maps->occ_words, maps->pitch_words, maps->rows, maps->cols, chrom_dev, parents_dev, n, n_waypoints,
        crossover_rate, mutation_rate, seeds_dev, (uint32_t)generation, children_dev);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

// ---------------------------------------------------------------------------------------------
// Population initialisers (pso.py:97-105, ga_solver.py:48-56, :95-104): the attempts of the reference's
// "generate -> evaluate -> accept if valid" loops, a batch at a time.  Attempt a draws from stream
// (seed, PSO_INIT / GA_INIT, 0, a), so a batch is any range of attempts and every rank can regenerate any of them.
// ---------------------------------------------------------------------------------------------
// PSO attempt: W waypoints [uniform(0, R-1), uniform(0, C-1)] (pso.py:50-51, draws 0..2W-1), then W velocities
// [uniform(-max_vel/5, max_vel/5)] x 2 (pso.py:105, draws 2W..4W-1); also the rounded, clamped cells (pso.py:61,69-70).
// Attempts [offsets[m], offsets[m] + n) of map m (offsets[m] < 0: the map is done, nothing is written).
__global__ void mpp_pso_init_kernel(int n, int W, const int32_t *__restrict__ offsets, int R, int C, double max_vel,
                                    const uint64_t *__restrict__ seeds, double *__restrict__ pos,
                                    double *__restrict__ vel, int32_t *__restrict__ wp_cells) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * W) return;
    const int attempt0 = offsets[blockIdx.y];
    if (attempt0 < 0) return;
    const uint64_t sd = seeds[blockIdx.y];
    const uint32_t k0 = (uint32_t)sd, k1 = (uint32_t)(sd >> 32);
    const size_t row = (size_t)blockIdx.y * n * W;
    pos += 2 * row; vel += 2 * row; wp_cells += row;
    const int p = t / W, dim = t % W;
    const uint32_t att = (uint32_t)(attempt0 + p);
    // draws 2*dim, 2*dim+1 = block dim; draws 2W + 2*dim, +1 = block W + dim
    const mpp_u4 a = mpp_philox((uint32_t)dim, att, 0u, MPP_CLS_PSO_INIT, k0, k1);
    const mpp_u4 b = mpp_philox((uint32_t)(W + dim), att, 0u, MPP_CLS_PSO_INIT, k0, k1);
    const double lo = -max_vel / 5, hi = max_vel / 5;
    const size_t i = ((size_t)p * W + dim) * 2;
    const double xr = 0 + ((double)(R - 1) - 0) * mpp_u53(a.x, a.y);   // random.uniform(a, b) = a + (b-a)*random()
    const double xc = 0 + ((double)(C - 1) - 0) * mpp_u53(a.z, a.w);
    pos[i] = xr; pos[i + 1] = xc;
    vel[i] = lo + (hi - lo) * mpp_u53(b.x, b.y);
    vel[i + 1] = lo + (hi - lo) * mpp_u53(b.z, b.w);
    int ir = (int)rint(xr), ic = (int)rint(xc);
    ir = max(0, min(R - 1, ir)); ic = max(0, min(C - 1, ic));
    wp_cells[(size_t)p * W + dim] = ir * C + ic;
}

extern "C" int mpp_pso_init_batch(const mpp_map_batch *maps, int n_attempts, const int32_t *attempt_offset_dev,
                                  int n_waypoints, double max_vel, const uint64_t *seeds_dev, double *pos_dev,
                                  double *vel_dev, int32_t *waypoint_cells_dev, void *stream) {
    MPP_REQUIRE(maps && attempt_offset_dev && seeds_dev && pos_dev && vel_dev && waypoint_cells_dev && n_attempts > 0 &&
                n_waypoints > 0 && maps->n_maps <= MPP_POP_MAX_MAPS, "mpp_pso_init_batch: bad argument");
    MPP_CUDA(cudaSetDevice(maps->device));
    const int total = n_attempts * n_waypoints;
    mpp_pso_init_kernel<<<dim3((total + 255) / 256, maps->n_maps), 256, 0, (cudaStream_t)stream>>>(
        n_attempts, n_waypoints, attempt_offset_dev, maps->rows, maps->cols, max_vel, seeds_dev, pos_dev, vel_dev,
        waypoint_cells_dev);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}

// GA attempt: W genes, each (randint(0, R-1), randint(0, C-1)) redrawn until the cell is free (ga_solver.py:48-56)
__global__ void mpp_ga_init_kernel(const uint32_t *__restrict__ occ, int occ_words, int pitch, int R, int C, int n, int W,
                                   const int32_t *__restrict__ offsets, const uint64_t *__restrict__ seeds,
                                   int32_t *__restrict__ chrom) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int attempt0 = offsets[blockIdx.y];
    if (attempt0 < 0) return;                                          // the map is done
    occ += (size_t)blockIdx.y * occ_words;
    chrom += (size_t)blockIdx.y * n * W;
    mpp_stream_rng rng;
    rng.init(seeds[blockIdx.y], MPP_CLS_GA_INIT, 0u, (uint32_t)(attempt0 + p));
    for (int k = 0; k < W; ++k) chrom[(size_t)p * W + k] = ga_random_free_cell(rng, occ, pitch, R, C);
}

extern "C" int mpp_ga_init_batch(const mpp_map_batch *maps, int n_attempts, const int32_t *attempt_offset_dev,
                                 int n_waypoints, const uint64_t *seeds_dev, int32_t *chrom_dev, void *stream) {
    MPP_REQUIRE(maps && attempt_offset_dev && seeds_dev && chrom_dev && n_attempts > 0 && n_waypoints > 0 &&
                maps->n_maps <= MPP_POP_MAX_MAPS, "mpp_ga_init_batch: bad argument");
    for (int k = 0; k < maps->n_maps; ++k)                             // the start cell is free: mutation terminates
        MPP_REQUIRE(maps->meta_host[k].start >= 0, "mpp_ga_init_batch: map %d has no start", k);
    MPP_CUDA(cudaSetDevice(maps->device));
    mpp_ga_init_kernel<<<dim3((n_attempts + 127) / 128, maps->n_maps), 128, 0, (cudaStream_t)stream>>>(
        maps->occ_dev, maps->occ_words, maps->pitch_words, maps->rows, maps->cols, n_attempts, n_waypoints,
        attempt_offset_dev, seeds_dev, chrom_dev);
    MPP_CUDA(cudaGetLastError());
    return MPP_OK;
}
