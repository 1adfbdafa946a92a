"""PSO / GA over batches of independent maps (PSOBatch, GABatch, mpp_waypoint_fitness_maps and the batched population
kernels) against the reference's recorded trajectories, the per-map solvers and the oracle mirrors.  Every comparison
is bit for bit: paths, statistics, Python types, convergence curves, evaluation and attempt counts."""
import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

INF = float("inf")
POLICY = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, min_safe_distance=1.8,
              diagonal_obstacle_penalty_value=100.0, allow_diagonal_moves=True,
              restrict_diagonal_near_obstacle_policy=True)
CASES = [(m, n) for m in ("fig7", "blocks40") for n in (20, 33)]


def _moved(grid, rng):
    """The map with start and target moved to two seeded random free cells."""
    g = np.where(grid >= 2, 0, grid)
    s, t = rng.choice(np.flatnonzero(g.ravel() == 0), 2, replace=False)
    g.flat[s], g.flat[t] = 2, 3
    return g


def _args(planner, K, N, W):
    return (K, N, W, 0.7, 1.5, 1.5) if planner == "pso" else (K, N, W, 0.1, 0.8, 3)


def _batch(planner, grids, K, N, W, seeds, **kw):
    from maaco_path_planing_b200.batch import GABatch, PSOBatch
    cls = PSOBatch if planner == "pso" else GABatch
    return cls(np.stack(grids), *_args(planner, K, N, W), seeds=seeds, **POLICY, **kw)


def _solo(planner, grid, K, N, W, seed):
    from maaco_path_planing_b200.ga_solver import GASolver
    from maaco_path_planing_b200.pso import PSOSolver
    cls = PSOSolver if planner == "pso" else GASolver
    s = cls(grid, *_args(planner, K, N, W), rng_seed=seed, verbose=False, **POLICY)
    return s, s.solve()


def _assert_same(got, solver, want, evals=None, attempts=None):
    assert got[:6] == tuple(want)
    assert [type(v) for v in got[:6]] == [type(v) for v in want]
    assert all(type(a) is int and type(b) is int for a, b in got[0])
    assert got[6] == solver.convergence_curve
    if evals is not None:
        assert evals == solver.fitness_evaluations
    if attempts is not None and hasattr(solver, "init_attempts"):
        assert attempts == solver.init_attempts


def _check_rows(planner, b, res, grids, K, N, W, seeds, rows=None):
    for m in (range(len(grids)) if rows is None else rows):
        s, want = _solo(planner, grids[m], K, N, W, seeds[m])
        _assert_same(res[m], s, want, b.fitness_evaluations[m], b.init_attempts[m])


@pytest.mark.parametrize("planner", ["pso", "ga"])
@pytest.mark.parametrize("name,N", CASES)
def test_golden_trajectory_as_a_row_of_a_wave(planner, name, N):
    g = load_golden("solver_cases")
    k = f"{planner}_{name}_{N}"
    _, K, seed = (int(x) for x in g[k + "_meta"])
    grid = g[k + "_grid"].astype(int)
    rng = np.random.default_rng(N)
    grids = [_moved(grid, rng), grid, _moved(grid, rng), _moved(grid, rng)]
    seeds = [seed + 1, seed, seed + 2, seed + 3]
    b = _batch(planner, grids, K, N, 5, seeds)
    res = b.solve()
    C = grid.shape[1]
    r = res[1]
    assert np.array_equal(np.array(r[6]), g[k + "_curve"])
    assert np.array_equal(np.array([p * C + q for p, q in r[0]], np.int32), g[k + "_best"])
    assert np.array_equal(np.array([float(x) for x in r[1:6]]), g[k + "_stats"])
    if planner == "pso":
        assert np.array_equal(b.pos[1].cpu().numpy(), g[k + "_pos"])
        assert np.array_equal(b.vel[1].cpu().numpy(), g[k + "_vel"])
        assert np.array_equal(b.pbest_fit[1].cpu().numpy(), g[k + "_pbest_fit"])
    else:
        assert np.array_equal(b.chrom[1].cpu().numpy(), g[k + "_chrom"])
        assert np.array_equal(b.fitness[1].cpu().numpy(), g[k + "_fit"])
    _check_rows(planner, b, res, grids, K, N, 5, seeds)


@pytest.mark.parametrize("planner", ["pso", "ga"])
@pytest.mark.parametrize("size,n_maps,N,K", [(64, 16, 256, 5), (100, 16, 96, 10)])
def test_maps_with_own_endpoints_equal_per_map_solvers(planner, size, n_maps, N, K):
    from maaco_path_planing_b200 import blocks_map
    rng = np.random.default_rng(size * 7 + N)
    grids = [_moved(blocks_map(size, 0.2, seed=300 + size + i), rng) for i in range(n_maps)]
    seeds = [1000 + 17 * i for i in range(n_maps)]
    b = _batch(planner, grids, K, N, 4, seeds)
    res = b.solve()
    _check_rows(planner, b, res, grids, K, N, 4, seeds)
    assert sum(len(r[0]) > 0 for r in res) == n_maps


@pytest.mark.parametrize("planner", ["pso", "ga"])
def test_fallback_failure_and_zero_waypoints_in_one_wave(planner):
    """The snake corridor (no waypoint chain is valid: the direct path is the one individual), its walled map (no path
    at all) and an open map in one wave; the same wave with W = 0 (one start -> target connector per map)."""
    g = load_golden("fallback_cases")
    N, K, seed = (int(x) for x in g[f"{planner}_meta"])
    open_map = np.zeros((9, 9), int)
    open_map[0, 0], open_map[8, 8] = 2, 3
    grids = [g["grid"].astype(int), g["walled_grid"].astype(int), open_map]
    seeds = [seed, 701, 9]
    for W in (5, 0):
        b = _batch(planner, grids, K, N, W, seeds)
        res = b.solve()
        _check_rows(planner, b, res, grids, K, N, W, seeds)
        assert res[1][:6] == ([], INF, 0, 0.0, 0.0, INF)
        assert len(res[0][0]) == len(g[f"{planner}_best"]) and len(res[2][0]) > 0


@pytest.mark.parametrize("planner", ["pso", "ga"])
def test_results_do_not_depend_on_waves_slots_or_buffer_sizes(planner):
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import solve_ga_batch, solve_pso_batch
    rng = np.random.default_rng(5)
    grids = [_moved(blocks_map(48, 0.2, seed=40 + i), rng) for i in range(7)]
    seeds = [77 + i for i in range(7)]
    K, N, W = 4, 40, 4
    if planner == "pso":
        sweep = lambda **kw: solve_pso_batch(grids, K, N, W, dict(w=0.7, c1=1.5, c2=1.5, **POLICY, **kw.pop("p", {})),
                                             seeds=seeds, **kw)
    else:
        sweep = lambda **kw: solve_ga_batch(grids, K, N, W, dict(mutation_rate=0.1, crossover_rate=0.8, **POLICY,
                                                                 **kw.pop("p", {})), seeds=seeds, **kw)
    base = sweep()
    assert [r[0] for r in base] == list(range(7))
    for wave in (1, 3):
        assert sweep(wave=wave) == base, wave
    for p in (dict(n_slots=5), dict(heap_cap=64), dict(max_cells=8)):
        assert sweep(p=p) == base, p
    b = _batch(planner, grids, K, N, W, seeds, max_cells=8, heap_cap=64)
    assert [r[:7] for r in b.solve()] == [r[1:] for r in base]
    assert b._search.max_cells > 8                                                     # grew and repeated


def test_two_maps_against_oracle_mirrors():
    from py_solvers import GaOracle, PsoOracle
    from maaco_path_planing_b200 import blocks_map
    rng = np.random.default_rng(11)
    grids = [_moved(blocks_map(56, 0.2, seed=61 + i), rng) for i in range(2)]
    N, K, W = 64, 4, 4
    b = _batch("pso", grids, K, N, W, [31, 32])
    res = b.solve()
    for m, g in enumerate(grids):
        o = PsoOracle(g, K, N, W, 0.7, 1.5, 1.5, 0.3, 0.8, 1.8, 100.0, 31 + m)
        opath, ofit = o.solve()
        assert res[m][6] == o.curve and res[m][5] == ofit
        assert [r * 56 + c for r, c in res[m][0]] == list(opath)
        assert np.array_equal(b.pos[m].cpu().numpy(), o.pos) and np.array_equal(b.vel[m].cpu().numpy(), o.vel)
        assert np.array_equal(b.pbest_fit[m].cpu().numpy(), o.pbest_fit)
    b = _batch("ga", grids, K, N, W, [41, 42])
    res = b.solve()
    for m, g in enumerate(grids):
        o = GaOracle(g, K, N, W, 0.1, 0.8, 3, 0.3, 0.8, 1.8, 100.0, 41 + m)
        opath, _ = o.solve()
        assert res[m][6] == o.curve
        assert [r * 56 + c for r, c in res[m][0]] == list(opath)
        assert np.array_equal(b.chrom[m].cpu().numpy(), np.array([ind[0] for ind in o.pop], np.int32))


@pytest.mark.parametrize("planner", ["pso", "ga"])
def test_config5_maps_equal_per_map_solvers(planner):
    """One wave of config-5 maps (blocks_map 256x256, 20% obstacles) at 256 individuals, 3 iterations, W = 5."""
    from maaco_path_planing_b200 import blocks_map
    grids = [blocks_map(256, 0.20, seed=5000 + i) for i in range(6)]
    seeds = [900 + i for i in range(6)]
    b = _batch(planner, grids, 3, 256, 5, seeds)
    res = b.solve()
    _check_rows(planner, b, res, grids, 3, 256, 5, seeds)


def test_sharded_sweep_two_gpus():
    """solve_pso_batch / solve_ga_batch with the maps sharded over 2 GPUs == the one-GPU sweep (skipped on a 1-GPU box)."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from conftest import ROOT
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29536", os.path.join(ROOT, "tests", "multigpu_pop_batch_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "multigpu_pop_batch_check ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
