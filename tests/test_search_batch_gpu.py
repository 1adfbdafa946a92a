"""A* / Dijkstra over batches of independent maps (SearchBatch, mpp_astar_batch_maps) against the reference's golden
vectors, the per-map solvers and the C oracle.  Everything is bit-exact: paths, g, statistics, Python types."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from test_oracle_golden import _astar_golden, _dijkstra_golden

pytestmark = pytest.mark.gpu

INF = float("inf")
EMPTY = ([], INF, 0, 0.0, 0.0, INF)


def _batch(grids, **kw):
    from maaco_path_planing_b200.batch import SearchBatch
    return SearchBatch(np.stack(grids), **kw)


def _moved(grid, rng):
    """The map with start and target moved to two seeded random free cells."""
    g = np.where(grid >= 2, 0, grid)
    s, t = rng.choice(np.flatnonzero(g.ravel() == 0), 2, replace=False)
    g.flat[s], g.flat[t] = 2, 3
    return g


def _random_queries(grids, per_map, rng, avoid_max=40):
    """per_map random (src, dst) cells of every map (obstacles included) and a random avoid set per query."""
    R, C = grids[0].shape
    n = len(grids) * per_map
    mi = np.repeat(np.arange(len(grids)), per_map).astype(np.int32)
    src = rng.integers(0, R * C, n).astype(np.int32)
    dst = rng.integers(0, R * C, n).astype(np.int32)
    dst[::7] = src[::7]
    avoid = np.zeros((n, (R * C + 31) // 32), np.uint32)
    for i in range(n):
        for c in rng.integers(0, R * C, int(rng.integers(0, avoid_max))):
            avoid[i, c >> 5] |= np.uint32(1 << (c & 31))
    return mi, src, dst, avoid


def _host(*ts):
    return [t.cpu().numpy() for t in ts]


def _grouped(cases, per_launch=8):
    """Cases grouped by (shape, allow_diagonal, restrict_corner), at most per_launch maps per batch."""
    groups = {}
    for c in cases:
        groups.setdefault((c[1].shape, c[5], c[6]), []).append(c)
    for (shape, ad, rs), cs in groups.items():
        for k in range(0, len(cs), per_launch):
            yield ad, rs, cs[k:k + per_launch]


def test_reference_goldens_as_map_batches():
    import pyoracle as O
    n_astar = n_dijkstra = 0
    for ad, rs, cs in _grouped(list(_astar_golden())):
        sb = _batch([c[1] for c in cs], allow_diagonal_moves=ad, restrict_diagonal_near_obstacle_policy=rs)
        bits = np.stack([O.cells_to_bits(c[4], c[1].size) for c in cs])
        mi, src, dst = np.arange(len(cs)), [c[2] for c in cs], [c[3] for c in cs]
        for variant, col in ((0, 7), (1, 8)):
            cells, ncell, g, _ = _host(*sb.search(variant, mi, src, dst, bits))
            for k, c in enumerate(cs):
                want = c[col]
                assert ncell[k] == len(want) and np.array_equal(cells[k, :ncell[k]], want), (c[0], variant)
                if variant == 1:
                    assert g[k] == c[9], (c[0], g[k], c[9])
        n_astar += len(cs)
    for ad, rs, cs in _grouped(list(_dijkstra_golden())):
        sb = _batch([c[1] for c in cs], allow_diagonal_moves=ad, restrict_diagonal_near_obstacle_policy=rs)
        bits = np.stack([O.cells_to_bits(c[4], c[1].size) for c in cs])
        cells, ncell, _, _ = _host(*sb.search(2, np.arange(len(cs)), [c[2] for c in cs], [c[3] for c in cs], bits))
        for k, c in enumerate(cs):
            assert ncell[k] == len(c[7]) and np.array_equal(cells[k, :ncell[k]], c[7]), c[0]
        n_dijkstra += len(cs)
    assert n_astar == 240 and n_dijkstra == 120


def _assert_same_as_solver(got, solver):
    want = solver.solve()
    assert got[:6] == want
    assert [type(v) for v in got[:6]] == [type(v) for v in want]
    assert all(type(a) is int and type(b) is int for a, b in got[0])
    assert solver.convergence_curve == ([] if got[6] is None else [got[6]])


@pytest.mark.parametrize("algorithm", ["astar", "dijkstra"])
def test_solve_equals_per_map_solvers(algorithm):
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.astar import AStarSolver
    from maaco_path_planing_b200.dijkstra import DijkstraSolver
    rng = np.random.default_rng(64)
    grids = [_moved(blocks_map(256, 0.2, seed=7000 + i), rng) for i in range(64)]
    res = _batch(grids).solve(algorithm)
    Solver = AStarSolver if algorithm == "astar" else DijkstraSolver
    for k, grid in enumerate(grids):
        _assert_same_as_solver(res[k], Solver(grid))
    assert sum(r[6] is not None for r in res) > 48


def test_dijkstra_fig7_anchor():
    """SURVEY 8(c), fig7 with main.py's policy: T=12, SP=0.3274397055203064, fitness=35.41830095052029."""
    from maaco_path_planing_b200.batch import solve_search_batch
    grid = load_golden("env_grids")["fig7"].astype(int)
    params = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, min_safe_distance=1.8,
                  diagonal_obstacle_penalty_value=100.0)
    (i, path, L, T, SP, DP, F, g), = solve_search_batch([grid], "dijkstra", params)
    assert i == 0 and len(path) == 28 and T == 12 and SP == 0.3274397055203064 and F == 35.41830095052029
    assert g is not None


@pytest.mark.parametrize("shape,n_maps,per_map", [((37, 42), 6, 10), ((100, 100), 4, 8), ((1000, 1000), 1, 3)])
def test_search_vs_oracle(shape, n_maps, per_map):
    """Several queries per map, each with its own avoid set, on maps that differ from each other; statistics for
    several min_safe_distance values (each rebuilds the batch's safety tables)."""
    import pyoracle as O
    from maaco_path_planing_b200.engine import make_policy
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    grids = [(rng.random(shape) < 0.25).astype(int) for _ in range(n_maps)]
    mi, src, dst, avoid = _random_queries(grids, per_map, rng)
    if shape[0] == 1000:                                   # long searches: endpoints on free cells in opposite corners
        free = [np.flatnonzero(g.ravel() == 0) for g in grids]
        src[:] = [f[f < 50 * 1000][int(rng.integers(0, 100))] for f in [free[m] for m in mi]]
        dst[:] = [f[f >= 950 * 1000][int(rng.integers(0, 100))] for f in [free[m] for m in mi]]
    sb = _batch(grids, turn_penalty_factor=0.3, safety_penalty_factor=0.8, diagonal_obstacle_penalty_value=100.0)
    orcs = [O.AStarOracle(g, True, True) for g in grids]
    n = len(mi)
    for variant in (0, 1, 2):
        want = [orcs[mi[i]].solve(variant, int(src[i]), int(dst[i]), avoid[i]) for i in range(n)]
        for msd in (0.0, 1.5, 3.2):
            sb.policy = make_policy(0.3, 0.8, msd, 100.0)
            e0 = sb.expansions()
            cells, ncell, g, stats = _host(*sb.search(variant, torch.as_tensor(mi).cuda(), torch.as_tensor(src).cuda(),
                                                      torch.as_tensor(dst).cuda(), avoid))
            assert sb.expansions() - e0 == sum(w[2] for w in want)
            for i in range(n):
                wc, wg = want[i][0], want[i][1]
                assert ncell[i] == len(wc) and np.array_equal(cells[i, :ncell[i]], wc), (variant, i)
                assert g[i] == wg, (variant, i, g[i], wg)
                if len(wc) and (grids[mi[i]].ravel()[wc] == 1).any():
                    # MPA.py:107-108 returns [src] for src == dst even on an obstacle; the safety classes (shared with
                    # mpp_path_stats) charge an obstacle's own cell nothing.  astar.py / dijkstra.py never return it.
                    assert variant == 1 and len(wc) == 1
                    continue
                ws = O.path_stats(grids[mi[i]], wc, 0.3, 0.8, msd, 100.0, True) if len(wc) else np.array(
                    [INF, 0, 0, 0, INF])
                assert np.array_equal(stats[i], ws), (variant, msd, i, stats[i], ws)
    assert (ncell > 1).sum() >= n // 3


def test_edge_cases():
    import pyoracle as O
    from maaco_path_planing_b200.astar import AStarSolver
    from maaco_path_planing_b200.dijkstra import DijkstraSolver
    enclosed = np.zeros((20, 20), int)
    enclosed[12:19, 12:19] = 1
    enclosed[13:18, 13:18] = 0
    enclosed[2, 2], enclosed[15, 15] = 2, 3
    side = np.zeros((20, 20), int)
    side[5, 4:9] = 1
    side[6, 6], side[6, 7] = 2, 3
    diag = np.zeros((20, 20), int)
    diag[9, 9], diag[10, 10] = 2, 3
    grids = [enclosed, side, diag]
    for algorithm, Solver in (("astar", AStarSolver), ("dijkstra", DijkstraSolver)):
        res = _batch(grids).solve(algorithm)
        assert res[0] == EMPTY + (None,)
        assert [type(v) for v in res[0][:6]] == [list, float, int, float, float, float]
        for k, grid in enumerate(grids):
            _assert_same_as_solver(res[k], Solver(grid))
        assert len(res[1][0]) == 2 and len(res[2][0]) == 2
    # start equal to target, invalid map indices and endpoints (not searched), next to valid queries
    sb = _batch(grids, turn_penalty_factor=0.3, safety_penalty_factor=0.8, diagonal_obstacle_penalty_value=100.0)
    s = 6 * 20 + 5
    mi = [1, 1, 3, -1, 0, 0, 2]
    src = [s, s, s, s, -1, 0, 0]
    dst = [s, s + 2, s, s, 0, 400, 399]
    for variant in (0, 1, 2):
        cells, ncell, g, stats = _host(*sb.search(variant, mi, src, dst))
        assert ncell[0] == 1 and cells[0, 0] == s and g[0] == 0.0
        assert np.array_equal(stats[0], O.path_stats(side, [s], 0.3, 0.8, 1.5, 100.0, True)) and stats[0, 0] == 0.0
        w, wg, _, _ = O.AStarOracle(side).solve(variant, s, s + 2)
        assert ncell[1] == len(w) and np.array_equal(cells[1, :ncell[1]], w) and g[1] == wg
        w, wg, _, _ = O.AStarOracle(diag).solve(variant, 0, 399)
        assert ncell[6] == len(w) and np.array_equal(cells[6, :ncell[6]], w) and g[6] == wg
        for i in (2, 3, 4, 5):
            assert ncell[i] == 0 and g[i] == INF and np.array_equal(stats[i], [INF, 0, 0, 0, INF])


def test_heap_overflow_and_truncation_grow():
    """A tiny heap (4-connected Dijkstra on open maps: every frontier cell at Manhattan distance d has g = d, so the
    ring's buckets overflow into the heap) and tiny path buffers grow and repeat the affected queries only; the
    results are the bytes of a roomy run."""
    grids = [np.zeros((100, 100), int) for _ in range(4)]
    grids[1][40:60, 30] = 1
    mi = np.repeat(np.arange(4), 3).astype(np.int32)
    src = np.array([0, 0, 5050] * 4, np.int32)
    dst = np.array([9999, 1, 5052] * 4, np.int32)
    kw = dict(allow_diagonal_moves=False)
    for variant, small, grown in ((0, dict(max_cells=4), "max_cells"), (2, dict(max_cells=4), "max_cells"),
                                  (2, dict(heap_cap=64), "heap_cap")):
        roomy = _batch(grids, **kw)
        want = _host(*roomy.search(variant, mi, src, dst))
        assert roomy.launches == 1
        sb = _batch(grids, **kw, **small)
        got = _host(*sb.search(variant, mi, src, dst))
        assert getattr(sb, grown) > small[grown] and sb.launches > 1, (variant, grown)
        for a, b in zip(got[1:], want[1:]):
            assert np.array_equal(a, b), (variant, grown)
        for i in range(len(mi)):
            assert np.array_equal(got[0][i, :got[1][i]], want[0][i, :want[1][i]]), (variant, grown, i)
        if grown == "heap_cap":
            assert int(sb.counters[3]) > 64                                  # the overflow heap was really used


def test_schedule_independence():
    """Same results whatever the number of search slots, the order in which they take the queries, and the waves."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import solve_search_batch
    rng = np.random.default_rng(17)
    grids = [_moved(blocks_map(64, 0.2, seed=900 + i), rng) for i in range(12)]
    mi, src, dst, avoid = _random_queries(grids, 6, rng)
    free = [np.flatnonzero(g.ravel() != 1) for g in grids]
    src[1::2] = [free[m][int(rng.integers(0, len(free[m])))] for m in mi[1::2]]
    dst[1::2] = [free[m][int(rng.integers(0, len(free[m])))] for m in mi[1::2]]
    ref = _batch(grids)
    want = _host(*ref.search(0, mi, src, dst, avoid))
    assert (want[1] > 1).sum() >= len(mi) // 3
    for n_slots in (1, 7, ref.max_slots):
        for longest_first in (True, False):
            sb = _batch(grids, n_slots=n_slots)
            got = _host(*sb.search(0, mi, src, dst, avoid, longest_first=longest_first))
            for a, b in zip(got[1:], want[1:]):
                assert np.array_equal(a, b), (n_slots, longest_first)
            for i in range(len(mi)):
                assert np.array_equal(got[0][i, :got[1][i]], want[0][i, :want[1][i]]), (n_slots, longest_first, i)
    for algorithm in ("astar", "dijkstra"):
        base = solve_search_batch(grids, algorithm, {})
        assert [r[0] for r in base] == list(range(len(grids)))
        for wave in (1, 3):
            assert solve_search_batch(grids, algorithm, {}, wave=wave) == base
