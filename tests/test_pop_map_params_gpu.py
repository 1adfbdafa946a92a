"""Per-map parameters of PSOBatch, GABatch and MPABatch (a parameter sweep as one wave: mpp_pso_update_batch_p,
mpp_ga_select_batch_p, mpp_ga_breed_batch_p, mpp_waypoint_fitness_maps_p, mpp_path_stats_p, mpp_mpa_init_batch_p,
mpp_mpa_iteration_batch_p) and of their sweeps.  Every row must equal the solo solver run with that row's parameters
and seed, bit for bit: paths, statistics, Python types, convergence curves, evaluation and attempt counts."""
import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _release_cached_memory():
    """Hand the waves' device memory back after each test: the config-5 waves leave tens of GB in torch's cache, which a
    later test that starts a fresh process would otherwise find taken."""
    yield
    import gc
    import torch
    gc.collect()
    torch.cuda.empty_cache()

INF = float("inf")
POLICY = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, min_safe_distance=1.8,
              diagonal_obstacle_penalty_value=100.0, allow_diagonal_moves=True,
              restrict_diagonal_near_obstacle_policy=True)
PSO_ARGS = dict(w=0.7, c1=1.5, c2=1.5)
GA_ARGS = dict(mutation_rate=0.1, crossover_rate=0.8, tournament_size=3)
MPA_PARAMS = dict(FADs_rate=0.2, P_const=0.5, levy_beta=2.0, turn_penalty_factor=0.1, safety_penalty_factor=0.8,
                  min_safe_distance=1.8, diagonal_obstacle_penalty=100.0)


def _moved(grid, rng):
    """The map with start and target moved to two seeded random free cells."""
    g = np.where(grid >= 2, 0, grid)
    s, t = rng.choice(np.flatnonzero(g.ravel() == 0), 2, replace=False)
    g.flat[s], g.flat[t] = 2, 3
    return g


def _assert_same(got, solver, want, evals=None, attempts=None):
    """(as tests/test_pop_batch_gpu.py compares a batch row with its solo solver)"""
    assert got[:6] == tuple(want)
    assert [type(v) for v in got[:6]] == [type(v) for v in want]
    assert all(type(a) is int and type(b) is int for a, b in got[0])
    assert got[6] == solver.convergence_curve
    if evals is not None:
        assert evals == solver.fitness_evaluations
    if attempts is not None and hasattr(solver, "init_attempts"):
        assert attempts == solver.init_attempts


def _varied(planner, M, W=4):
    """One parameter set per map, every per-map key varied (GA: tournament sizes 2..5, and 7 for the last map)."""
    out = []
    for m in range(M):
        p = dict(turn_penalty_factor=0.05 * (m % 5), safety_penalty_factor=0.2 + 0.3 * (m % 4),
                 diagonal_obstacle_penalty_value=(10.0, 100.0, 1000.0)[m % 3])
        if planner == "pso":
            p.update(w=0.4 + 0.1 * (m % 6), c1=1.0 + 0.25 * (m % 3), c2=2.0 - 0.25 * (m % 4))
        else:
            p.update(mutation_rate=0.05 * (1 + m % 4), crossover_rate=0.5 + 0.1 * (m % 5),
                     tournament_size=7 if m == M - 1 else 2 + m % 4)
        out.append(p)
    return out


def _batch(planner, grids, K, N, W, seeds, map_params=None, **kw):
    from maaco_path_planing_b200.batch import GABatch, PSOBatch
    if planner == "pso":
        return PSOBatch(np.stack(grids), K, N, W, **PSO_ARGS, seeds=seeds, map_params=map_params, **POLICY, **kw)
    return GABatch(np.stack(grids), K, N, W, **GA_ARGS, seeds=seeds, map_params=map_params, **POLICY, **kw)


def _solo(planner, grid, K, N, W, seed, params):
    from maaco_path_planing_b200.ga_solver import GASolver
    from maaco_path_planing_b200.pso import PSOSolver
    if planner == "pso":
        s = PSOSolver(grid, K, N, W, rng_seed=seed, verbose=False, **{**PSO_ARGS, **POLICY, **params})
    else:
        s = GASolver(grid, K, N, W, rng_seed=seed, verbose=False, **{**GA_ARGS, **POLICY, **params})
    return s, s.solve()


def _check_rows(planner, b, res, grids, K, N, W, seeds, map_params, rows=None):
    for m in (range(len(grids)) if rows is None else rows):
        s, want = _solo(planner, grids[m], K, N, W, seeds[m], map_params[m] if map_params else {})
        _assert_same(res[m], s, want, b.fitness_evaluations[m], b.init_attempts[m])


@pytest.mark.parametrize("planner", ["pso", "ga"])
@pytest.mark.parametrize("size,N,K", [(64, 256, 5), (100, 96, 8)])
def test_every_row_equals_its_solo_solver(planner, size, N, K):
    """16 maps with their own endpoints, every per-map key varied (GA: population > 85 so that tournaments of 7 run)."""
    from maaco_path_planing_b200 import blocks_map
    M = 16
    rng = np.random.default_rng(size * 3 + N)
    grids = [_moved(blocks_map(size, 0.2, seed=800 + size + i), rng) for i in range(M)]
    seeds = [2000 + 13 * i for i in range(M)]
    mp = _varied(planner, M)
    b = _batch(planner, grids, K, N, 4, seeds, mp)
    assert b.map_params[3] == {**b.map_params[3], **mp[3]}
    res = b.solve()
    _check_rows(planner, b, res, grids, K, N, 4, seeds, mp)
    assert sum(len(r[0]) > 0 for r in res) == M


@pytest.mark.parametrize("planner", ["pso", "ga"])
def test_golden_trajectory_as_a_row_of_a_per_map_wave(planner):
    g = load_golden("solver_cases")
    k = f"{planner}_fig7_33"
    _, K, seed = (int(x) for x in g[k + "_meta"])
    grid = g[k + "_grid"].astype(int)
    rng = np.random.default_rng(33)
    grids = [_moved(grid, rng), grid, _moved(grid, rng)]
    seeds = [seed + 1, seed, seed + 2]
    mp = _varied(planner, 3)
    mp[-1]["tournament_size" if planner == "ga" else "w"] = 2 if planner == "ga" else 0.3
    mp[1] = {}                                                    # the golden row: the wave's own parameters
    b = _batch(planner, grids, K, 33, 5, seeds, mp)
    res = b.solve()
    C = grid.shape[1]
    assert np.array_equal(np.array(res[1][6]), g[k + "_curve"])
    assert np.array_equal(np.array([p * C + q for p, q in res[1][0]], np.int32), g[k + "_best"])
    assert np.array_equal(np.array([float(x) for x in res[1][1:6]]), g[k + "_stats"])
    if planner == "pso":
        assert np.array_equal(b.pos[1].cpu().numpy(), g[k + "_pos"])
        assert np.array_equal(b.pbest_fit[1].cpu().numpy(), g[k + "_pbest_fit"])
    else:
        assert np.array_equal(b.chrom[1].cpu().numpy(), g[k + "_chrom"])
        assert np.array_equal(b.fitness[1].cpu().numpy(), g[k + "_fit"])
    _check_rows(planner, b, res, grids, K, 33, 5, seeds, mp)


@pytest.mark.parametrize("planner", ["pso", "ga"])
def test_config5_wave_sampled_rows(planner):
    """32 config-5 maps (256x256, 20% obstacles), 1024 individuals, 2 iterations, a parameter set per map."""
    from maaco_path_planing_b200 import blocks_map
    M = 32
    grids = [blocks_map(256, 0.20, seed=5000 + i) for i in range(M)]
    seeds = [700 + i for i in range(M)]
    mp = _varied(planner, M)
    b = _batch(planner, grids, 2, 1024, 5, seeds, mp)
    res = b.solve()
    _check_rows(planner, b, res, grids, 2, 1024, 5, seeds, mp, rows=(0, 13, 30, 31))


@pytest.mark.parametrize("planner", ["pso", "ga"])
def test_fallback_and_zero_waypoint_waves_take_map_weights(planner):
    """The snake corridor (its one individual is the direct path), its walled map and an open map under per-map
    weights; the same wave with W = 0 (one start -> target connector and mpp_path_stats_p per map)."""
    g = load_golden("fallback_cases")
    N, K, seed = (int(x) for x in g[f"{planner}_meta"])
    open_map = np.zeros((9, 9), int)
    open_map[0, 0], open_map[8, 8] = 2, 3
    grids = [g["grid"].astype(int), g["walled_grid"].astype(int), open_map]
    seeds = [seed, 701, 9]
    mp = [dict(turn_penalty_factor=1.5, diagonal_obstacle_penalty_value=7.0), {"safety_penalty_factor": 2.0},
          dict(turn_penalty_factor=0.01, safety_penalty_factor=0.0)]
    for W in (5, 0):
        b = _batch(planner, grids, K, N, W, seeds, mp)
        res = b.solve()
        _check_rows(planner, b, res, grids, K, N, W, seeds, mp)
        assert res[1][:6] == ([], INF, 0, 0.0, 0.0, INF)


@pytest.mark.parametrize("planner", ["pso", "ga"])
def test_empty_mappings_equal_no_map_params(planner):
    """map_params=[{}] * M runs the per-map kernels with the constructor's values: byte for byte the default wave."""
    from maaco_path_planing_b200 import blocks_map
    rng = np.random.default_rng(4)
    grids = [_moved(blocks_map(48, 0.2, seed=90 + i), rng) for i in range(5)]
    seeds = [5 + i for i in range(5)]
    a = _batch(planner, grids, 4, 64, 4, seeds)
    b = _batch(planner, grids, 4, 64, 4, seeds, [{}] * 5)
    ra, rb = a.solve(), b.solve()
    assert repr(ra) == repr(rb)
    assert a.fitness_evaluations == b.fitness_evaluations and a.init_attempts == b.init_attempts
    if planner == "pso":
        assert a.pos.cpu().numpy().tobytes() == b.pos.cpu().numpy().tobytes()
        assert a.pbest_fit.cpu().numpy().tobytes() == b.pbest_fit.cpu().numpy().tobytes()
    else:
        assert a.chrom.cpu().numpy().tobytes() == b.chrom.cpu().numpy().tobytes()
        assert a.fitness.cpu().numpy().tobytes() == b.fitness.cpu().numpy().tobytes()


@pytest.mark.parametrize("planner", ["pso", "ga"])
def test_buffer_growth_keeps_the_parameters(planner):
    from maaco_path_planing_b200 import blocks_map
    rng = np.random.default_rng(6)
    grids = [_moved(blocks_map(48, 0.2, seed=140 + i), rng) for i in range(4)]
    seeds = [61 + i for i in range(4)]
    mp = _varied(planner, 4)
    mp[-1]["tournament_size" if planner == "ga" else "w"] = 4 if planner == "ga" else 0.2
    b = _batch(planner, grids, 4, 40, 4, seeds, mp, max_cells=8, heap_cap=64)
    res = b.solve()
    assert b._search.max_cells > 8                                                     # grew and repeated
    _check_rows(planner, b, res, grids, 4, 40, 4, seeds, mp)


# ---- MPA ---------------------------------------------------------------------------------------------------------------

def _mpa_solo(grid, N, K, seed, params):
    from maaco_path_planing_b200.mpa import MPA
    s = MPA(grid, num_predators=N, num_iterations=K, rng_seed=seed, verbose=False, **params)
    return tuple(s.solve_path_planning()) + (s.convergence_curve_data,)


def _mpa_varied(M):
    return [dict(FADs_rate=(0.1, 0.2, 0.35)[m % 3], P_const=0.3 + 0.1 * (m % 4), levy_beta=(1.2, 1.5, 2.0)[m % 3],
                 turn_penalty_factor=0.05 * (m % 4), safety_penalty_factor=0.5 * (m % 2),
                 diagonal_obstacle_penalty=(10.0, 100.0, 1000.0)[(m + 1) % 3], min_safe_distance=1.0 + m)
            for m in range(M)]


def test_mpa_rows_equal_solo_mpa_and_the_oracle():
    from py_solvers import MpaOracle
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MPABatch
    M, N, K = 8, 256, 6
    rng = np.random.default_rng(8)
    grids = [_moved(blocks_map(64, 0.2, seed=660 + i), rng) for i in range(M)]
    seeds = [31 + i for i in range(M)]
    mp = _mpa_varied(M)
    res = MPABatch(np.stack(grids), N, K, seeds=seeds, map_params=mp, **MPA_PARAMS).solve()
    for i in range(M):
        assert res[i] == _mpa_solo(grids[i], N, K, seeds[i], {**MPA_PARAMS, **mp[i]}), i
    for i in (0, 5):
        p = {**MPA_PARAMS, **mp[i]}
        o = MpaOracle(grids[i], N, K, p["FADs_rate"], p["P_const"], p["levy_beta"], p["turn_penalty_factor"],
                      p["safety_penalty_factor"], p["min_safe_distance"], p["diagonal_obstacle_penalty"], seeds[i])
        opath, ost = o.solve()
        assert res[i][6] == o.curve and [r * 64 + c for r, c in res[i][0]] == list(opath) and res[i][5] == ost[4], i
    # map_params of empty mappings: the default wave, byte for byte
    assert repr(MPABatch(np.stack(grids), N, K, seeds=seeds, map_params=[{}] * M, **MPA_PARAMS).solve()) == \
        repr(MPABatch(np.stack(grids), N, K, seeds=seeds, **MPA_PARAMS).solve())


def test_mpa_overflow_repeat_keeps_the_parameters():
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MPABatch
    M, N, K = 4, 64, 6
    grids = [blocks_map(64, 0.2, seed=690 + i) for i in range(M)]
    seeds = [41 + i for i in range(M)]
    mp = _mpa_varied(M)
    want = [_mpa_solo(grids[i], N, K, seeds[i], {**MPA_PARAMS, **mp[i]}) for i in range(M)]
    for kw in (dict(heap_cap=64), dict(max_cells=16)):
        b = MPABatch(np.stack(grids), N, K, seeds=seeds, map_params=mp, **kw, **MPA_PARAMS)
        assert b.solve() == want, kw


# ---- sweeps ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("planner", ["pso", "ga", "mpa"])
@pytest.mark.parametrize("on_device", [False, True])
def test_sweeps_over_two_shapes_split_waves_by_per_wave_keys(planner, on_device):
    import torch
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import solve_ga_batch, solve_mpa_batch, solve_pso_batch
    rng = np.random.default_rng(12)
    grids = [_moved(blocks_map(40 if i % 2 else 48, 0.2, seed=300 + i), rng) for i in range(8)]
    seeds = [400 + i for i in range(8)]
    K, N, W = 3, 48, 3
    if planner == "mpa":
        mp = [dict(m, allow_diagonal_moves=i != 3) for i, m in enumerate(_mpa_varied(8))]
    else:
        mp = [dict(m, min_safe_distance=2.5 if i in (2, 6) else 1.8, allow_diagonal_moves=i != 5)
              for i, m in enumerate(_varied(planner, 8))]
        if planner == "ga":
            mp[7]["tournament_size"] = 5                          # (a population of 48 takes tournaments up to 5)
    src = [torch.as_tensor(g, device="cuda") for g in grids] if on_device else grids
    if planner == "pso":
        out = solve_pso_batch(src, K, N, W, dict(PSO_ARGS, **POLICY), seeds=seeds, wave=3, map_params=mp)
    elif planner == "ga":
        out = solve_ga_batch(src, K, N, W, dict(GA_ARGS, **POLICY), seeds=seeds, wave=3, map_params=mp)
    else:
        out = solve_mpa_batch(src, N, K, MPA_PARAMS, seeds=seeds, wave=3, map_params=mp)
    assert [r[0] for r in out] == list(range(8))
    for i, g in enumerate(grids):
        if planner == "mpa":
            assert out[i][1:] == _mpa_solo(g, N, K, seeds[i], {**MPA_PARAMS, **mp[i]}), i
        else:
            s, want = _solo(planner, g, K, N, W, seeds[i], mp[i])
            _assert_same(out[i][1:], s, want)


def test_side_stream():
    """A per-map wave enqueued on a side stream of torch gives the default stream's results."""
    import torch
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MPABatch
    rng = np.random.default_rng(21)
    grids = [_moved(blocks_map(48, 0.2, seed=500 + i), rng) for i in range(3)]
    seeds = [3, 4, 5]
    mp, mpa = _varied("ga", 3), _mpa_varied(3)
    mp[-1]["tournament_size"] = 5
    want = _batch("ga", grids, 3, 40, 3, seeds, mp).solve(), \
        MPABatch(np.stack(grids), 64, 4, seeds=seeds, map_params=mpa, **MPA_PARAMS).solve()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = _batch("ga", grids, 3, 40, 3, seeds, mp).solve(), \
            MPABatch(np.stack(grids), 64, 4, seeds=seeds, map_params=mpa, **MPA_PARAMS).solve()
    s.synchronize()
    assert got == want
