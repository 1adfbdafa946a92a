"""The search, fitness and MPA kernels on both sides of their shared-memory staging limits, against the oracle.

mpp_astar_batch_maps and mpp_waypoint_fitness_maps on a one-map batch, and mpp_mpa_iteration_batch on any batch, stage
a map's packed occupancy in dynamic shared memory up to 32 KB without the opt-in attribute, up to 40 KB with it, and
read it through L2 above that.  The kernels
also declare ~16 KB of static shared memory, so a map of exactly 32 KB of occupancy needs the opt-in too.  Raising
the attribute lasts for the rest of the process, so the 32 KB maps are only tested honestly in a process in which no
larger map ran before: run as a script, this file checks the 32 KB shapes first and only then a larger one, and prints
`smem_tiers_check ok`.  tests/test_smem_tiers_gpu.py runs it that way and imports its checks for the other tiers.
    python tests/smem_tiers_check.py
"""
import functools
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

# (rows, cols, occupancy bytes, tier); occupancy bytes = 4 * (((rows + 2) * ceil((cols + 2) / 32) + 3) & ~3)
SHAPES = [
    (480, 480, 30848, "staged"),
    (500, 500, 32128, "staged"),
    (510, 510, 32768, "staged, at the limit"),
    (1022, 254, 32768, "staged, at the limit"),
    (254, 1022, 32768, "staged, at the limit"),
    (511, 511, 34896, "first opt-in"),
    (566, 566, 40896, "last opt-in"),
    (567, 567, 40976, "first global"),
]
AT_LIMIT = [s[:2] for s in SHAPES if s[2] == 32768]

FIT_POLICY = (0.3, 0.8, 1.8, 100.0)            # main.py's PSO / GA policy (tpf, spf, msd, diagonal penalty)
SOLVER_POLICY = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, min_safe_distance=1.8,
                     diagonal_obstacle_penalty_value=100.0, allow_diagonal_moves=True,
                     restrict_diagonal_near_obstacle_policy=True)
MPA_PARAMS = dict(FADs_rate=0.2, P_const=0.5, levy_beta=1.5, turn_penalty_factor=0.1, safety_penalty_factor=0.8,
                  min_safe_distance=1.8, diagonal_obstacle_penalty=100.0)
MPA_N, MPA_K = 32, 3                           # 3 iterations: one of each phase


@functools.lru_cache(maxsize=None)
def grid_of(rows, cols, k=0):
    """The k-th test map of a shape: 20% block obstacles, start (0, 0), target (rows-1, cols-1)."""
    from maaco_path_planing_b200 import blocks_map
    g = blocks_map(0, 0.2, seed=100000 * k + 1000 * rows + cols, rows=rows, cols=cols)
    g.setflags(write=False)
    return g


def cells_of(path, cols):
    return [r * cols + c for r, c in path]


def _engine(grid):
    from maaco_path_planing_b200 import GridMap
    from maaco_path_planing_b200.engine import SearchEngine
    return SearchEngine(GridMap(grid))


def check_occ_bytes(rows, cols, want):
    """The map layout still puts this shape at `want` bytes of occupancy (else the shape no longer tests its tier)."""
    from maaco_path_planing_b200 import GridMap
    _, pitch = GridMap(grid_of(rows, cols)).occ_bits()
    assert 4 * (((rows + 2) * pitch + 3) & ~3) == want, (rows, cols, pitch, want)


def _queries(grid, n, rng):
    """n connector queries: corner to corner both ways, src == dst, obstacle endpoints, random free pairs; per-query
    avoid sets (none, random cells, a wall across the middle row with one gap)."""
    R, C = grid.shape
    flat = grid.ravel()
    free, obst = np.flatnonzero(flat != 1), np.flatnonzero(flat == 1)
    src = free[rng.integers(0, len(free), n)].astype(np.int32)
    dst = free[rng.integers(0, len(free), n)].astype(np.int32)
    src[0], dst[0] = 0, R * C - 1
    src[1], dst[1] = R * C - 1, 0
    src[2], dst[2] = free[C + 7], (R - 1) * C + C // 3
    dst[3] = src[3]
    src[4] = obst[0]
    dst[5] = obst[len(obst) // 2]
    avoid = np.zeros((n, (R * C + 31) // 32), np.uint32)

    def mark(i, cells):
        for c in cells:
            avoid[i, c >> 5] |= np.uint32(1 << (c & 31))

    for i in range(8, n, 2):                                  # random cells, sometimes an endpoint among them
        mark(i, rng.integers(0, R * C, int(rng.integers(1, 400))))
    for i in range(9, n, 4):                                  # a wall across the middle row, one gap
        gap = int(rng.integers(0, C))
        mark(i, [(R // 2) * C + c for c in range(C) if c != gap])
    mark(6, [0, 1, C, C + 1])                                 # corner to corner with the start's neighbours avoided
    src[6], dst[6] = 0, R * C - 1
    return src, dst, avoid


def check_connectors(grid, n=48, seed=0):
    """SearchEngine.astar_batch, variants 0 (A*), 1 (MPA's connector), 2 (Dijkstra) == AStarOracle.solve: path,
    n_cells, g and the summed node expansions."""
    import pyoracle as O
    R, C = grid.shape
    src, dst, avoid = _queries(grid, n, np.random.default_rng(seed))
    eng = _engine(grid)
    orc = O.AStarOracle(grid, True, True)
    for variant in (0, 1, 2):
        eng.counters.zero_()
        cells, ncell, g = eng.astar_batch(variant, src, dst, avoid.view(np.int32), True, True)
        cells, ncell, g = cells.cpu().numpy(), ncell.cpu().numpy(), g.cpu().numpy()
        expansions = 0
        for i in range(n):
            want, wg, e, _ = orc.solve(variant, int(src[i]), int(dst[i]), avoid[i])
            expansions += e
            assert ncell[i] == len(want), (variant, i, ncell[i], len(want))
            assert np.array_equal(cells[i, :ncell[i]], want), (variant, i)
            assert g[i] == wg or (np.isinf(g[i]) and np.isinf(wg)), (variant, i, g[i], wg)
        assert eng.expansions()[0] == expansions, (variant, eng.expansions()[0], expansions)
        assert ncell[0] >= max(R, C) and ncell[3] == 1 and ncell[4] == 0 and ncell[5] == 0, variant


def check_fitness(grid, N=96, W=3, seed=0, stats_modes=False):
    """SearchEngine.waypoint_fitness == the oracle's: cells, n_cells, statistics, expansions.  With `stats_modes`, also
    mpp_path_stats of those paths in both statistics modes, up to the largest supported safety distance (180)."""
    import pyoracle as O
    from maaco_path_planing_b200.engine import make_policy
    R, C = grid.shape
    rng = np.random.default_rng(seed)
    wps = rng.integers(0, R * C, (N, W)).astype(np.int32)                  # PSO-style: may hit obstacles
    free = np.flatnonzero(grid.ravel() != 1)
    wps[N // 4:] = free[rng.integers(0, len(free), (N - N // 4, W))]        # GA-style: free cells
    wps[5, 1] = wps[5, 0]                                                   # repeated waypoint
    wps[6, 0] = 0                                                           # waypoint on the start
    eng = _engine(grid)
    dcells, dncell, dstats = eng.waypoint_fitness(wps, make_policy(*FIT_POLICY))
    cells, ncell, stats = dcells.cpu().numpy(), dncell.cpu().numpy(), dstats.cpu().numpy()
    ocells, oncell, ostats, oexp = O.waypoint_fitness(grid, wps, *FIT_POLICY, threads=0)
    assert np.array_equal(ncell, oncell)
    for i in range(N):
        assert np.array_equal(cells[i, :ncell[i]], ocells[i, :oncell[i]]), i
    assert np.array_equal(stats, ostats)
    assert eng.expansions()[0] == oexp
    assert N // 3 < (ncell > 0).sum() < N                                   # valid and invalid individuals
    if not stats_modes:
        return
    for mode, tpf in ((0, 0.3), (1, 0.1)):
        for msd in (0.0, 1.8, 23.7, 180.0):
            st = eng.path_stats(dcells, dncell, make_policy(tpf, 0.8, msd, 100.0, mode=mode)).cpu().numpy()
            # the oracle scans a (2 msd + 3)^2 box per cell: at msd 180 in mode 0, every 3rd path
            rows = range(0, N, 3) if (mode, msd) == (0, 180.0) else range(N)
            for i in rows:
                want = O.path_stats(grid, cells[i, :ncell[i]], tpf, 0.8, msd, 100.0, True, mode=mode)
                assert np.array_equal(st[i], want), (mode, msd, i, st[i], want)


def _mpa_solo(grid, seed):
    from maaco_path_planing_b200.mpa import MPA
    s = MPA(grid, num_predators=MPA_N, num_iterations=MPA_K, rng_seed=seed, verbose=False, **MPA_PARAMS)
    return s, tuple(s.solve_path_planning()) + (s.convergence_curve_data,)


def check_mpa(grid, seed=7):
    """Solo MPA == MpaOracle: the curve, the best path and fitness, every predator's final path."""
    from py_solvers import MpaOracle
    p = MPA_PARAMS
    s, res = _mpa_solo(grid, seed)
    o = MpaOracle(grid, MPA_N, MPA_K, p["FADs_rate"], p["P_const"], p["levy_beta"], p["turn_penalty_factor"],
                  p["safety_penalty_factor"], p["min_safe_distance"], p["diagonal_obstacle_penalty"], seed)
    opath, ost = o.solve()
    C = grid.shape[1]
    assert res[6] == o.curve
    assert cells_of(res[0], C) == list(opath) and res[5] == ost[4]
    cells, ncell = s._pop["cells"].cpu().numpy(), s._pop["ncell"].cpu().numpy()
    for i, ind in enumerate(o.pop):
        assert np.array_equal(cells[i, :ncell[i]], np.array(ind["path"], np.int32)), f"predator {i}"
    return res


def check_mpa_batch(rows, cols, seeds=(7, 8, 9), first=None):
    """MPABatch over 3 maps of one shape == solo MPA map by map (`first`: the solo result of map 0, if known)."""
    from maaco_path_planing_b200.batch import MPABatch
    grids = [grid_of(rows, cols, k) for k in range(len(seeds))]
    res = MPABatch(np.stack(grids), MPA_N, MPA_K, seeds=list(seeds), **MPA_PARAMS).solve()
    for k, g in enumerate(grids):
        want = first if (k == 0 and first is not None) else _mpa_solo(g, seeds[k])[1]
        assert res[k] == want, (rows, cols, k)


def check_pso_ga(grid, N=32, K=2, W=3):
    """PSOSolver / GASolver == the oracle's mirrors of their solve loops."""
    from py_solvers import GaOracle, PsoOracle
    from maaco_path_planing_b200.ga_solver import GASolver
    from maaco_path_planing_b200.pso import PSOSolver
    C = grid.shape[1]
    s = PSOSolver(grid, num_iterations=K, num_particles=N, num_waypoints_per_particle=W, w=0.7, c1=1.5, c2=1.5,
                  rng_seed=31, verbose=False, **SOLVER_POLICY)
    res = s.solve()
    o = PsoOracle(grid, K, N, W, 0.7, 1.5, 1.5, *FIT_POLICY, 31)
    opath, ofit = o.solve()
    assert s.convergence_curve == o.curve and res[5] == ofit
    assert cells_of(res[0], C) == list(opath) and len(opath) > 0
    assert np.array_equal(s._state["pos"].cpu().numpy(), o.pos) and np.array_equal(s._state["vel"].cpu().numpy(), o.vel)
    assert np.array_equal(s._state["pbest_fit"].cpu().numpy(), o.pbest_fit)
    ga = GASolver(grid, num_generations=K, population_size=N, num_waypoints_per_chromosome=W, mutation_rate=0.1,
                  crossover_rate=0.8, tournament_size=3, rng_seed=32, verbose=False, **SOLVER_POLICY)
    gres = ga.solve()
    go = GaOracle(grid, K, N, W, 0.1, 0.8, 3, *FIT_POLICY, 32)
    gpath, gst = go.solve()
    assert ga.convergence_curve == go.curve and gres[5] == gst[4]
    assert cells_of(gres[0], C) == list(gpath) and len(gpath) > 0
    assert np.array_equal(ga._pop["chrom"].cpu().numpy(), np.array([ind[0] for ind in go.pop], np.int32))


def check_shape(rows, cols, want_bytes, stats_modes=False):
    """Every check of one shape: the three launchers (A*/Dijkstra, fitness, MPA solo and batched)."""
    check_occ_bytes(rows, cols, want_bytes)
    g = grid_of(rows, cols)
    check_connectors(g)
    check_fitness(g, stats_modes=stats_modes)
    check_mpa_batch(rows, cols, first=check_mpa(g))


def main():
    import torch
    torch.cuda.set_device(0)
    done = []
    for rows, cols, nbytes, _ in SHAPES:                      # every 32 KB shape before any larger map
        if nbytes == 32768:
            check_shape(rows, cols, nbytes, stats_modes=(rows, cols) == (510, 510))
            done.append(f"{rows}x{cols}")
    check_pso_ga(grid_of(510, 510))
    big = next(s for s in SHAPES if s[2] > 32768)
    check_shape(*big[:3])                                     # raises the kernels' limits ...
    check_connectors(grid_of(510, 510), seed=1)               # ... which must not change a 32 KB map's results
    print(f"smem_tiers_check ok: {', '.join(done)} (32 KB, first in the process), 510x510 PSO / GA, "
          f"then {big[0]}x{big[1]} and 510x510 again")


if __name__ == "__main__":
    main()
