"""Whole-solver parity: PSOSolver / GASolver (CUDA update + fitness kernels, host control flow)
against trajectories recorded from the unmodified reference under the injected Philox streams.
Waypoints, positions, chosen individuals and paths bit-exact; fitness / stats bit-exact fp64."""
import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

POLICY = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, min_safe_distance=1.8,
              diagonal_obstacle_penalty_value=100.0, allow_diagonal_moves=True,
              restrict_diagonal_near_obstacle_policy=True)
CASES = [(m, n) for m in ("fig7", "blocks40") for n in (20, 33)]


@pytest.mark.parametrize("name,N", CASES)
def test_pso_trajectory(name, N):
    from maaco_path_planing_b200.pso import PSOSolver
    g = load_golden("solver_cases")
    k = f"pso_{name}_{N}"
    _, K, seed = (int(x) for x in g[k + "_meta"])
    grid = g[k + "_grid"].astype(int)
    s = PSOSolver(grid, num_iterations=K, num_particles=N, num_waypoints_per_particle=5, w=0.7, c1=1.5, c2=1.5,
                  rng_seed=seed, verbose=False, **POLICY)
    assert s._initialize_particles()
    S = s._state
    assert np.array_equal(S["pos"].cpu().numpy(), g[k + "_init_pos"])
    assert np.array_equal(S["vel"].cpu().numpy(), g[k + "_init_vel"])
    assert np.array_equal(S["cur_stats"][:, 4].cpu().numpy(), g[k + "_init_fit"])
    s2 = PSOSolver(grid, num_iterations=K, num_particles=N, num_waypoints_per_particle=5, w=0.7, c1=1.5, c2=1.5,
                   rng_seed=seed, verbose=False, **POLICY)
    res = s2.solve()
    assert np.array_equal(np.array(s2.convergence_curve), g[k + "_curve"])
    C = grid.shape[1]
    assert np.array_equal(np.array([r * C + c for r, c in res[0]], np.int32), g[k + "_best"])
    assert np.array_equal(np.array([float(x) for x in res[1:]]), g[k + "_stats"])
    S = s2._state
    assert np.array_equal(S["pos"].cpu().numpy(), g[k + "_pos"])          # every particle, bit-exact after K iterations
    assert np.array_equal(S["vel"].cpu().numpy(), g[k + "_vel"])
    assert np.array_equal(S["pbest_fit"].cpu().numpy(), g[k + "_pbest_fit"])
    assert np.array_equal(S["cur_stats"][:, 4].cpu().numpy(), g[k + "_cur_fit"])
    parts = s2.particles
    assert len(parts) == N and parts[0]["pbest_path"][0] == s2.start_node


@pytest.mark.parametrize("name,N", CASES)
def test_ga_trajectory(name, N):
    from maaco_path_planing_b200.ga_solver import GASolver
    g = load_golden("solver_cases")
    k = f"ga_{name}_{N}"
    _, K, seed = (int(x) for x in g[k + "_meta"])
    grid = g[k + "_grid"].astype(int)
    mk = lambda: GASolver(grid, num_generations=K, population_size=N, num_waypoints_per_chromosome=5, mutation_rate=0.1,
                          crossover_rate=0.8, tournament_size=3, rng_seed=seed, verbose=False, **POLICY)
    s = mk()
    assert s._initialize_population()
    assert np.array_equal(s._pop["chrom"].cpu().numpy(), g[k + "_init_chrom"])
    assert np.array_equal(s._pop["stats"][:, 4].cpu().numpy(), g[k + "_init_fit"])
    s2 = mk()
    res = s2.solve()
    assert np.array_equal(np.array(s2.convergence_curve), g[k + "_curve"])
    C = grid.shape[1]
    assert np.array_equal(np.array([r * C + c for r, c in res[0]], np.int32), g[k + "_best"])
    assert np.array_equal(np.array([float(x) for x in res[1:]]), g[k + "_stats"])
    assert np.array_equal(s2._pop["chrom"].cpu().numpy(), g[k + "_chrom"])  # final population, sorted order
    assert np.array_equal(s2._pop["stats"][:, 4].cpu().numpy(), g[k + "_fit"])
    pop = s2.population
    assert len(pop) == N and pop[0]["path"][-1] == s2.target_node


def test_astar_solver_dropin_matches_reference_anchor():
    """SURVEY 8(c) anchor: A* on fig7 with main.py's policy -> 28 cells, L=31.556349186104047, T=17,
    SP=0.34870130201414323, fitness=36.93531022771536 (values printed by the unmodified reference)."""
    from maaco_path_planing_b200.astar import AStarSolver
    grid = load_golden("env_grids")["fig7"].astype(int)
    a = AStarSolver(grid, **POLICY)
    path, L, T, SP, DP, F = a.solve()
    assert len(path) == 28 and L == 31.556349186104047 and T == 17
    assert SP == 0.34870130201414323 and DP == 0.0 and F == 36.93531022771536
    assert a.convergence_curve == [L] or abs(a.convergence_curve[0] - L) < 1e-9
    p2, *_ = a.solve(start_node_override=(3, 3), target_node_override=(3, 3))
    assert p2 == [(3, 3)]
    assert a.solve(start_node_override=(0, 4), target_node_override=(5, 5))[0] == []   # obstacle start


def test_solver_errors_like_reference():
    from maaco_path_planing_b200.ga_solver import GASolver
    from maaco_path_planing_b200.pso import PSOSolver
    g = np.zeros((6, 6), int)
    with pytest.raises(ValueError, match="PSO: Start node not found."):
        PSOSolver(g, 2, 4, 2, 0.7, 1.5, 1.5)
    with pytest.raises(ValueError, match="GA: Start node not found."):
        GASolver(g, 2, 4, 2, 0.1, 0.8)


def test_fallback_individuals_match_reference(capsys):
    """pso.py:128-145 / ga_solver.py:111-117: when none of the N*20 random waypoint chains is feasible the reference
    carries on with ONE individual built from the direct start -> target path; pso.py:147-157 /
    ga_solver.py:120-126: no path at all -> ([], inf, 0, 0.0, 0.0, inf).  Recorded from the reference on a
    one-cell-wide snake corridor (tests/golden/make_golden.py::fallback_cases)."""
    from maaco_path_planing_b200.ga_solver import GASolver
    from maaco_path_planing_b200.pso import PSOSolver
    g = load_golden("fallback_cases")
    grid = g["grid"].astype(int)
    C = grid.shape[1]
    N, K, seed = (int(x) for x in g["pso_meta"])
    s = PSOSolver(grid, K, N, 5, 0.7, 1.5, 1.5, rng_seed=seed, verbose=False, **POLICY)
    res = s.solve()
    assert "PSO Warning: Population init failed, used a direct A* path as one particle." in capsys.readouterr().out
    assert [r * C + c for r, c in res[0]] == g["pso_best"].tolist()
    assert np.array_equal(np.array([float(x) for x in res[1:]]), g["pso_stats"])
    assert np.array_equal(np.array(s.convergence_curve), g["pso_curve"])
    assert np.array_equal(np.array([p["position"] for p in s.particles], dtype=float), g["pso_pos"])
    assert np.array_equal(np.array([p["current_fitness"] for p in s.particles]), g["pso_cur_fit"])
    N, K, seed = (int(x) for x in g["ga_meta"])
    s = GASolver(grid, K, N, 5, 0.1, 0.8, 3, rng_seed=seed, verbose=False, **POLICY)
    res = s.solve()
    assert "GA Warning: Population init failed, used a direct A* path as one individual." in capsys.readouterr().out
    assert [r * C + c for r, c in res[0]] == g["ga_best"].tolist()
    assert np.array_equal(np.array([float(x) for x in res[1:]]), g["ga_stats"])
    assert np.array_equal(np.array(s.convergence_curve), g["ga_curve"])
    assert np.array_equal(np.array([ind["fitness"] for ind in s.population]), g["ga_fit"])
    assert all(ind["chromosome"] == [] for ind in s.population)
    walled = g["walled_grid"].astype(int)
    r1 = PSOSolver(walled, 2, 2, 3, 0.7, 1.5, 1.5, rng_seed=701, verbose=False, **POLICY).solve()
    r2 = GASolver(walled, 2, 2, 3, 0.1, 0.8, rng_seed=702, verbose=False, **POLICY).solve()
    for r, want in ((r1, g["walled_pso_stats"]), (r2, g["walled_ga_stats"])):
        assert r[0] == [] and np.array_equal(np.array([float(x) for x in r[1:]]), want)


@pytest.mark.parametrize("name,N", [(m, n) for m in ("fig7", "blocks40") for n in (20, 24)])
def test_mpa_trajectory(name, N):
    """MPA: phases 1-3 (Brownian / Levy targets, private-A* reconstruction), memory, FADs, sorts and the
    best cascade vs the reference.  Paths bit-exact; fitness bit-exact fp64.  (The Kinderman-Monahan
    accept test uses the device log(): a draw within ~1 ulp of the boundary could differ -- p < 1e-12.)"""
    from maaco_path_planing_b200.mpa import MPA
    g = load_golden("solver_cases")
    k = f"mpa_{name}_{N}"
    _, K, seed, beta10 = (int(x) for x in g[k + "_meta"])
    grid = g[k + "_grid"].astype(int)
    s = MPA(grid, num_predators=N, num_iterations=K, FADs_rate=0.2, P_const=0.5, levy_beta=beta10 / 10.0,
            turn_penalty_factor=0.1, safety_penalty_factor=0.8, min_safe_distance=1.8, diagonal_obstacle_penalty=100.0,
            allow_diagonal_moves=True, restrict_diagonal_near_obstacle=True, rng_seed=seed, verbose=False)
    res = s.solve_path_planning()
    curve = np.array([np.inf if v is None else v for v in s.convergence_curve_data])
    assert np.array_equal(curve, g[k + "_curve"])
    C = grid.shape[1]
    assert np.array_equal(np.array([r * C + c for r, c in res[0]], np.int32), g[k + "_best"])
    assert np.array_equal(np.array([float(x) for x in res[1:]]), g[k + "_stats"])
    assert np.array_equal(s._pop["stats"][:, 4].cpu().numpy(), g[k + "_pop_fit"])
    offs = g[k + "_pop_offs"]
    cells, ncell = s._pop["cells"].cpu().numpy(), s._pop["ncell"].cpu().numpy()
    for i in range(N):
        assert np.array_equal(cells[i, :ncell[i]], g[k + "_pop_cells"][offs[i]:offs[i + 1]]), f"predator {i}"


def test_mpa_batched_maps_equal_individual_solves():
    """Config-5 style sweep: MPA over several independent maps in one launch per iteration (device-side stable sorts read
    through an index, best cascade vectorised over the maps) returns exactly what MPA returns map by map -- and the
    golden-pinned single-map run is among them."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MPABatch, solve_mpa_batch
    from maaco_path_planing_b200.mpa import MPA
    g = load_golden("solver_cases")
    k = "mpa_blocks40_24"
    N, K, seed, beta10 = (int(x) for x in g[k + "_meta"])
    kw = dict(FADs_rate=0.2, P_const=0.5, levy_beta=beta10 / 10.0, turn_penalty_factor=0.1, safety_penalty_factor=0.8,
              min_safe_distance=1.8, diagonal_obstacle_penalty=100.0)
    grids = [g[k + "_grid"].astype(int)] + [blocks_map(40, 0.2, seed=60 + i) for i in range(3)]
    seeds = [seed, 11, 12, 13]
    b = MPABatch(np.stack(grids), N, K, seeds=seeds, **kw)
    res = b.solve()
    for i, (path, length, turns, sp, dp, fit, curve) in enumerate(res):
        solo = MPA(grids[i], N, K, rng_seed=seeds[i], verbose=False, **kw)
        want = solo.solve_path_planning()
        assert (path, length, turns, sp, dp, fit) == tuple(want), i
        assert curve == solo.convergence_curve_data, i
    assert np.array_equal(np.array([r * 40 + c for r, c in res[0][0]], np.int32), g[k + "_best"])
    assert np.array_equal(np.array(res[0][6], dtype=float), g[k + "_curve"])
    # the sweep helper: maps of two shapes, waves of 2
    mixed = grids + [blocks_map(24, 0.2, seed=70)]
    out = solve_mpa_batch(mixed, 16, 4, kw, seeds=[5, 6, 7, 8, 9], wave=2)
    assert [r[0] for r in out] == [0, 1, 2, 3, 4]
    for r in out:
        solo = MPA(mixed[r[0]], 16, 4, rng_seed=[5, 6, 7, 8, 9][r[0]], verbose=False, **kw)
        assert tuple(r[1:7]) == tuple(solo.solve_path_planning()) and r[7] == solo.convergence_curve_data
    # tiny path buffers / heaps: the solve notices on the device and repeats itself with more room
    small = MPABatch(np.stack(grids[:2]), 12, 3, seeds=[1, 2], max_cells=16, heap_cap=64, **kw)
    big = MPABatch(np.stack(grids[:2]), 12, 3, seeds=[1, 2], **kw)
    assert small.solve() == big.solve()


def test_mpa_anchor_and_errors():
    """SURVEY 8(c): the initial MPA population on fig7 is the private-A* S->T path: 28 cells,
    L=31.556349186104047, fitness = L + 0.1*turns."""
    from maaco_path_planing_b200.mpa import MPA
    grid = load_golden("env_grids")["fig7"].astype(int)
    s = MPA(grid, 8, 3, levy_beta=2.0, turn_penalty_factor=0.1, safety_penalty_factor=0.8, min_safe_distance=1.8,
            diagonal_obstacle_penalty=100.0, rng_seed=1, verbose=False)
    ind = s.population[0]
    assert len(ind["path"]) == 28 and ind["length"] == 31.556349186104047 and ind["safety_penalty"] == 0.0
    assert ind["fitness"] == ind["length"] + 0.1 * ind["turns"]
    with pytest.raises(ValueError, match="MPA: Start node not found in grid."):
        MPA(np.zeros((5, 5), int), 4, 2)


def test_demo_driver_runs_all_planners(tmp_path):
    """The main.py-equivalent driver: all six planners on one map, results exported to .npz."""
    import subprocess
    import sys
    from conftest import ROOT
    out = tmp_path / "demo.npz"
    r = subprocess.run([sys.executable, "-m", "maaco_path_planing_b200.demo", "--map", "blocks:40:1", "--scale", "0.1",
                        "--out", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    z = np.load(out)
    for name in ("MAACO", "MPA", "A*", "Dijkstra", "GA", "PSO"):
        p = z[name + "_path"]
        assert len(p) > 0 and tuple(p[0]) == (0, 0) and tuple(p[-1]) == (39, 39), name
    assert z["A*_stats"][0] <= z["GA_stats"][0] + 1e-9                     # A* length is optimal


def test_pso_ga_medium_vs_oracle_mirrors():
    """Sizes beyond the recorded reference goldens: the CUDA solvers vs the oracle's sequential mirrors of the
    solve loops (themselves pinned to the reference in tests/test_oracle_golden.py)."""
    from py_solvers import GaOracle, PsoOracle
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.ga_solver import GASolver
    from maaco_path_planing_b200.pso import PSOSolver
    g = blocks_map(72, 0.2, seed=61)
    N, K = 96, 4
    s = PSOSolver(g, num_iterations=K, num_particles=N, num_waypoints_per_particle=4, w=0.7, c1=1.5, c2=1.5,
                  rng_seed=31, verbose=False, **POLICY)
    res = s.solve()
    o = PsoOracle(g, K, N, 4, 0.7, 1.5, 1.5, 0.3, 0.8, 1.8, 100.0, 31)
    opath, ofit = o.solve()
    assert s.convergence_curve == o.curve and res[5] == ofit
    assert [r * 72 + c for r, c in res[0]] == list(opath)
    assert np.array_equal(s._state["pos"].cpu().numpy(), o.pos) and np.array_equal(s._state["vel"].cpu().numpy(), o.vel)
    assert np.array_equal(s._state["pbest_fit"].cpu().numpy(), o.pbest_fit)
    ga = GASolver(g, num_generations=K, population_size=N, num_waypoints_per_chromosome=4, mutation_rate=0.1,
                  crossover_rate=0.8, tournament_size=3, rng_seed=32, verbose=False, **POLICY)
    gres = ga.solve()
    go = GaOracle(g, K, N, 4, 0.1, 0.8, 3, 0.3, 0.8, 1.8, 100.0, 32)
    gpath, gst = go.solve()
    assert ga.convergence_curve == go.curve
    assert [r * 72 + c for r, c in gres[0]] == list(gpath)
    assert np.array_equal(ga._pop["chrom"].cpu().numpy(), np.array([ind[0] for ind in go.pop], np.int32))


def test_population_kernels_one_map_batch_full_size_vs_oracle():
    """K8 / K9 at BASELINE config-3 population (4096 x 5 waypoints, 512x512): update, selection and breeding
    kernels on a one-map batch vs the C oracle, bit-exact."""
    import ctypes as C
    import torch
    import pyoracle as O
    from maaco_path_planing_b200 import _lib, GridMap, blocks_map
    g = blocks_map(512, 0.2, seed=3512)
    gm = GridMap(g)
    dev = torch.device("cuda", gm.device)
    L = _lib.lib()
    N, W, seed, it = 4096, 5, 77, 3
    rng = np.random.default_rng(0)
    pos = rng.random((N, W, 2)) * 511
    vel = (rng.random((N, W, 2)) - 0.5) * 30
    pbest = rng.random((N, W, 2)) * 511
    gbest = rng.random((W, 2)) * 511
    d_pos, d_vel = torch.as_tensor(pos.copy(), device=dev), torch.as_tensor(vel.copy(), device=dev)
    d_pb, d_gb = torch.as_tensor(pbest, device=dev), torch.as_tensor(gbest, device=dev)
    wp = torch.empty((N, W), dtype=torch.int32, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    max_vel = max(1.0, 0.15 * 512)
    seeds = torch.tensor([seed], dtype=torch.int64, device=dev)
    first = torch.zeros(1, dtype=torch.int32, device=dev)                  # every particle
    _lib.check(L.mpp_pso_update_batch(gm.handle, _lib.ptr(d_pos), _lib.ptr(d_vel), _lib.ptr(d_pb), _lib.ptr(d_gb), N,
                                      _lib.ptr(first), W, 0.7, 1.5, 1.5, max_vel, _lib.ptr(seeds), it, _lib.ptr(wp),
                                      stream), "mpp_pso_update_batch")
    torch.cuda.synchronize()
    owp = np.zeros(W, np.int32)
    gpos, gvel, gwp = d_pos.cpu().numpy(), d_vel.cpu().numpy(), wp.cpu().numpy()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for i in list(range(0, N, 37)) + [N - 1]:
        a, b = np.ascontiguousarray(pos[i]), np.ascontiguousarray(vel[i])
        O.lib().orc_pso_update_particle(p(a), p(b), p(np.ascontiguousarray(pbest[i])), p(gbest), W, C.c_double(0.7),
                                        C.c_double(1.5), C.c_double(1.5), C.c_double(max_vel), 512, 512, C.c_uint64(seed),
                                        it, i, p(owp))
        assert np.array_equal(gpos[i], a) and np.array_equal(gvel[i], b) and np.array_equal(gwp[i], owp), i
    # selection + breeding
    fit = np.sort(rng.random(N) * 100 + 700)
    d_fit = torch.as_tensor(fit, device=dev)
    parents = torch.empty(N, dtype=torch.int32, device=dev)
    _lib.check(L.mpp_ga_select_batch(gm.handle, _lib.ptr(d_fit), N, 3, _lib.ptr(seeds), it, _lib.ptr(parents), stream),
               "mpp_ga_select_batch")
    free = np.flatnonzero(g.ravel() != 1)
    chrom = free[rng.integers(0, len(free), (N, W))].astype(np.int32)
    d_chrom = torch.as_tensor(chrom, device=dev)
    children = torch.empty((N, W), dtype=torch.int32, device=dev)
    _lib.check(L.mpp_ga_breed_batch(gm.handle, _lib.ptr(d_chrom), _lib.ptr(parents), N, W, 0.8, 0.1, _lib.ptr(seeds), it,
                                    _lib.ptr(children), stream), "mpp_ga_breed_batch")
    torch.cuda.synchronize()
    par, ch = parents.cpu().numpy(), children.cpu().numpy()
    want = np.array([O.lib().orc_ga_select(p(fit), N, 3, C.c_uint64(seed), it, t) for t in range(N)], np.int32)
    assert np.array_equal(par, want)
    g8 = np.ascontiguousarray(g, dtype=np.uint8)
    c1, c2 = np.zeros(W, np.int32), np.zeros(W, np.int32)
    for pair in range(N // 2):
        O.lib().orc_ga_breed_pair(p(g8), 512, 512, p(np.ascontiguousarray(chrom[par[2 * pair]])),
                                  p(np.ascontiguousarray(chrom[par[2 * pair + 1]])), W, C.c_double(0.8), C.c_double(0.1),
                                  C.c_uint64(seed), it, pair, p(c1), p(c2))
        assert np.array_equal(ch[2 * pair], c1) and np.array_equal(ch[2 * pair + 1], c2), pair


@pytest.mark.parametrize("beta", [2.0, 1.5])
def test_mpa_medium_vs_oracle_mirror(beta):
    """MPA beyond the recorded goldens: 128 predators x 9 iterations on a 72x72 map vs the oracle's mirror of the
    solve loop (libm transcendental functions on the oracle side, device ones in the kernel)."""
    from py_solvers import MpaOracle
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.mpa import MPA
    g = blocks_map(72, 0.2, seed=62)
    N, K, seed = 128, 9, 41
    s = MPA(g, num_predators=N, num_iterations=K, FADs_rate=0.2, P_const=0.5, levy_beta=beta, turn_penalty_factor=0.1,
            safety_penalty_factor=0.8, min_safe_distance=1.8, diagonal_obstacle_penalty=100.0, rng_seed=seed, verbose=False)
    res = s.solve_path_planning()
    o = MpaOracle(g, N, K, 0.2, 0.5, beta, 0.1, 0.8, 1.8, 100.0, seed)
    opath, ost = o.solve()
    assert s.convergence_curve_data == o.curve
    assert [r * 72 + c for r, c in res[0]] == list(opath) and res[5] == ost[4]
    cells, ncell = s._pop["cells"].cpu().numpy(), s._pop["ncell"].cpu().numpy()
    for i, ind in enumerate(o.pop):
        assert np.array_equal(cells[i, :ncell[i]], np.array(ind["path"], np.int32)), f"predator {i}"


def test_sharded_populations_two_gpus():
    """PSO / GA / MPA with their populations sharded over 2 GPUs == reference goldens (skipped on a 1-GPU box)."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from conftest import ROOT
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29534", os.path.join(ROOT, "tests", "multigpu_solvers_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "multigpu_solvers_check ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
