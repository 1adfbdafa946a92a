"""Batched map sweeps (batch.py) at the launch shapes of BASELINE config 5 -- waves of 128 256x256 maps with 1024 ants,
device buffers handed from wave to wave, 1024-predator MPA populations -- against the per-map solvers and the C oracle.
Everything is bit-exact: per-ant records, pheromone fields, paths, lengths, turns, fitness and convergence curves."""
import numpy as np
import pytest

from conftest import MAACO_DEFAULT

INF = float("inf")
# main.py:44-52, the MPA parameters bench.py's config-5 MPA part runs with
MPA_PARAMS = dict(FADs_rate=0.2, P_const=0.5, levy_beta=2.0, turn_penalty_factor=0.1, safety_penalty_factor=0.8,
                  min_safe_distance=1.8, diagonal_obstacle_penalty=100.0)
ORACLE_MAPS = (0, 1, 63, 64, 126, 127)          # first / last map of a wave and both sides of its middle


def serpentine(n=48):
    """One-cell-wide corridor: rows 1, 3, ... are walls with one gap at alternating ends, start (0, 0), target at the
    corridor's end (n-2, 0).  The only path visits every free cell: 1175 cells at n = 48."""
    g = np.zeros((n, n), np.int64)
    for k, r in enumerate(range(1, n, 2)):
        g[r, :] = 1
        if r < n - 1:
            g[r, n - 1 if k % 2 == 0 else 0] = 0
    g[0, 0] = 2
    g[n - 2, 0 if (n // 2 - 1) % 2 else n - 1] = 3
    return g


def with_endpoints(g, start, target):
    """`g` with its start and target moved to the given cells (their 2x2 corners cleared, like blocks_map's)."""
    g = g.copy()
    g[(g == 2) | (g == 3)] = 0
    for (r, c), v in ((start, 2), (target, 3)):
        r0, c0 = min(r, g.shape[0] - 2), min(c, g.shape[1] - 2)
        g[r0:r0 + 2, c0:c0 + 2] = 0
        g[r, c] = v
    return g


def walled_in(g):
    """`g` with its start (0, 0) boxed in by obstacles: no ant can leave it."""
    g = g.copy()
    g[0, 1] = g[1, 0] = g[1, 1] = 1
    return g


def solo_solve(grid, N, K, seed, **kw):
    """What MAACO returns and stores for one map: (path, length, turns, convergence_curve)."""
    from maaco_path_planing_b200 import MAACO
    m = MAACO(grid, N, K, rng_seed=seed, verbose=False, **MAACO_DEFAULT, **kw)
    path, length, turns = m.solve_path_planning()
    return path, length, turns, m.convergence_curve_data


def cells_of(path, cols):
    return [r * cols + c for r, c in path]


def assert_equals_oracle(res, orc, cols):
    """A (path, length, turns, curve) of MAACOBatch == MaacoOracle.solve() of the same map and seed."""
    path, length, turns, curve = res
    opath, olen, oturns = orc.solve()
    assert cells_of(path, cols) == opath.tolist()
    assert length == olen and turns == (oturns if oturns >= 0 else INF)
    assert curve == orc.curve


def test_serpentine_best_path_outgrows_default_max_cells():
    """The long-path tests below only test something while the serpentine's best path is longer than the default path
    capacity of MAACO / MAACOBatch."""
    import pyoracle as O
    from maaco_path_planing_b200.batch import default_max_cells
    g = serpentine()
    path, length, turns = O.MaacoOracle(g, 8, 1, seed=1, threads=0, **MAACO_DEFAULT).solve()
    assert len(path) == int((g != 1).sum()) == 1175 and length == 1174.0
    assert len(path) - 1 > default_max_cells(*g.shape)


# ---- MAACO -----------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_config5_wave_vs_solo_and_oracle(monkeypatch):
    """One bench-sized wave: 128 256x256 maps x 1024 ants, the tour kernel at 16 ants per warp with grid.y = 128.  Two
    passes and the rest of the solve, map by map against solo MAACO (which runs the same colony at 2 ants per warp) and
    on six maps against the C oracle."""
    import torch
    import pyoracle as O
    from maaco_path_planing_b200 import MAACO, blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    monkeypatch.delenv("MPP_TOUR_APW", raising=False)
    M, N, K = 128, 1024, 3
    # a copy of the automatic ants-per-warp rule of tours_launch (csrc/mpp_maaco.cu, "ants per warp"), which the ABI does
    # not report: halve from 16 while the launch would have fewer than 12 warps per SM.  Change both together.
    sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    apw = 16
    while apw > 2 and -(-N * M // apw) < 12 * sm:
        apw >>= 1
    assert apw == 16
    grids = np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(M)])
    seeds = list(range(M))
    b = MAACOBatch(grids, N, K, seeds=seeds, **MAACO_DEFAULT)
    assert b.n_maps == M and b._apw == 0
    passes = []
    for it in (1, 2):
        b.run_iteration(it)
        passes.append(b.last_results() + (b.pheromone(),))
    res = b.solve()
    nc = passes[1][0]
    assert (nc > 0).mean() > 0.5                                          # most tours reach the target
    assert sum(1 for r in res if r[0]) == M
    for i in range(M):
        solo = MAACO(grids[i], N, K, rng_seed=seeds[i], verbose=False, **MAACO_DEFAULT)
        orc = O.MaacoOracle(grids[i], N, K, seed=seeds[i], threads=0, **MAACO_DEFAULT) if i in ORACLE_MAPS else None
        for it, (bnc, bln, btn, btau) in enumerate(passes, 1):
            solo.run_iteration(it)
            snc, sln, stn = solo.last_results()
            assert np.array_equal(bnc[i], snc) and np.array_equal(bln[i], sln) and np.array_equal(btn[i], stn), (i, it)
            assert np.array_equal(btau[i], solo.pheromone_matrix), (i, it)
            if orc is not None:
                _, onc, oln, otn, _ = orc.iterate(it)
                assert np.array_equal(bnc[i], onc) and np.array_equal(bln[i], oln) and np.array_equal(btn[i], otn), (i, it)
                assert np.array_equal(btau[i].ravel(), orc.tau), (i, it)
        path, length, turns = solo.solve_path_planning()
        assert res[i] == (path, length, turns, solo.convergence_curve_data), i
        if orc is not None:
            orc.iterate(3)
            assert cells_of(res[i][0], 256) == orc.best_path.tolist() and res[i][1] == orc.best_len, i
            assert res[i][3] == orc.curve, i


@pytest.mark.gpu
def test_reused_buffers_across_waves():
    """bench.py's chain of waves: a warm-up wave left after one pass hands its device buffers to the next wave of other
    maps, whose full solve hands them on to a third.  Each reused wave == a wave on fresh buffers, pass by pass, and
    == solo MAACO.  A walled-in map in a reused wave must not pick up the previous wave's best path or log."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    M, N, K = 6, 1024, 3
    maps = [blocks_map(256, 0.20, seed=5000 + i) for i in range(3 * M)]
    maps[M + 2] = walled_in(maps[M + 2])
    maps[2 * M + 4] = walled_in(maps[2 * M + 4])
    wave = lambda w, **kw: MAACOBatch(np.stack(maps[w * M:(w + 1) * M]), N, K, seeds=list(range(w * M, (w + 1) * M)),
                                      **MAACO_DEFAULT, **kw)
    prev = wave(0)
    prev.run_iteration(1)
    for w in (1, 2):
        b = wave(w, reuse=prev)
        for name in ("_tau", "_slabs", "_moves", "_best_cells", "_log"):
            assert getattr(b, name).data_ptr() == getattr(prev, name).data_ptr(), name
        fresh = wave(w)
        assert fresh._tau.data_ptr() != b._tau.data_ptr()
        for it in range(1, K + 1):
            b.run_iteration(it)
            fresh.run_iteration(it)
            for x, y in zip(b.last_results(), fresh.last_results()):
                assert np.array_equal(x, y), (w, it)
            assert np.array_equal(b.pheromone(), fresh.pheromone()), (w, it)
        res = b.solve()
        assert res == fresh.solve()
        for k in range(M):
            i = w * M + k
            assert res[k] == solo_solve(maps[i], N, K, i), i
        walled = 2 if w == 1 else 4
        assert res[walled] == ([], INF, INF, [None] * K)
        assert all(r[0] for k, r in enumerate(res) if k != walled)
        prev.close()
        fresh.close()
        prev = b


@pytest.mark.gpu
def test_solve_maaco_batch_groups_endpoints_into_ragged_waves(monkeypatch):
    """solve_maaco_batch on maps of three (start, target) pairs, interleaved, in groups of 7, 8 and 4 with waves of 3:
    every group ends with a ragged wave and its full waves run on the previous wave's buffers; every result == solo."""
    from maaco_path_planing_b200 import MppError, blocks_map
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch
    ends = [((0, 0), (63, 63)), ((0, 63), (63, 0)), ((63, 63), (0, 0))]
    labels = [0, 1, 2] * 4 + [0, 1, 0, 1, 0, 1, 1]                            # groups of 7, 8 and 4 maps
    grids = [with_endpoints(blocks_map(64, 0.20, seed=700 + i), *ends[e]) for i, e in enumerate(labels)]
    seeds = [40 + i for i in range(len(grids))]
    seen = []

    class Recording(batch.MAACOBatch):
        def __init__(self, grids, *args, reuse=None, **kw):
            super().__init__(grids, *args, reuse=reuse, **kw)
            seen.append((self.n_maps, reuse is not None and self._moves.data_ptr() == reuse._moves.data_ptr()))

    monkeypatch.setattr(batch, "MAACOBatch", Recording)
    N, K = 128, 3
    res = solve_maaco_batch(grids, N, K, MAACO_DEFAULT, seeds=seeds, wave=3)
    assert seen == [(3, False), (3, True), (1, False),                      # group 0: 7 maps
                    (3, False), (3, True), (2, False),                      # group 1: 8 maps
                    (3, False), (1, False)]                                 # group 2: 4 maps
    assert [r[0] for r in res] == list(range(len(grids)))
    for i, path, length, turns, curve in res:
        assert (path, length, turns, curve) == solo_solve(grids[i], N, K, seeds[i]), i
        assert path and path[0] == ends[labels[i]][0] and path[-1] == ends[labels[i]][1]
    # one wave cannot hold maps of different endpoints: it shares their tables
    with pytest.raises(MppError, match="mpp_maaco_tables.*must share start and target"):
        batch.MAACOBatch(np.stack(grids[:2]), N, K, seeds=seeds[:2], **MAACO_DEFAULT)


@pytest.mark.gpu
def test_truncated_move_buffers_do_not_reach_tau():
    """An explicit max_cells far below the tour lengths: moves past it are dropped, but every per-ant record and the
    pheromone field (built from the visited sets, not from the moves) stay exactly the oracle's; the solve then raises
    because the best path cannot be returned and the capacity was the caller's choice."""
    import pyoracle as O
    from maaco_path_planing_b200 import MppError, blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    grids = [blocks_map(96, 0.20, seed=96 + i) for i in range(2)]
    N, K = 256, 3
    b = MAACOBatch(np.stack(grids), N, K, seeds=[5, 6], max_cells=64, **MAACO_DEFAULT)
    orcs = [O.MaacoOracle(g, N, K, seed=s, threads=0, **MAACO_DEFAULT) for g, s in zip(grids, (5, 6))]
    for it in range(1, K + 1):
        b.run_iteration(it)
        nc, ln, tn = b.last_results()
        tau = b.pheromone()
        for k, orc in enumerate(orcs):
            _, onc, oln, otn, _ = orc.iterate(it)
            assert np.array_equal(nc[k], onc) and np.array_equal(ln[k], oln) and np.array_equal(tn[k], otn), (k, it)
            assert np.array_equal(tau[k].ravel(), orc.tau), (k, it)
        assert (nc - 1 > 64).mean() > 0.5                                      # most tours really were cut
    with pytest.raises(MppError, match="outgrew max_cells=64"):
        b.solve()


@pytest.mark.gpu
def test_best_path_longer_than_default_max_cells(monkeypatch):
    """A best path longer than the default path capacity (the serpentine's 1175 cells against 1024): MAACOBatch and
    solve_maaco_batch repeat the wave with full capacity and return what MAACO and the oracle return, like MAACO
    itself; with the capacity given explicitly the solve raises."""
    import pyoracle as O
    from maaco_path_planing_b200 import MppError, blocks_map
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import MAACOBatch, default_max_cells, solve_maaco_batch
    ends = ((0, 0), (46, 0))
    grids = [serpentine()] + [with_endpoints(blocks_map(48, 0.20, seed=480 + i), *ends) for i in range(4)]
    seeds = [11, 12, 13, 14, 15]
    N, K = 32, 3
    want = [solo_solve(g, N, K, s) for g, s in zip(grids, seeds)]
    for g, s, r in zip(grids, seeds, want):
        assert_equals_oracle(r, O.MaacoOracle(g, N, K, seed=s, threads=0, **MAACO_DEFAULT), 48)
    assert len(want[0][0]) == 1175 and all(r[0] for r in want)
    b = MAACOBatch(np.stack(grids[:3]), N, K, seeds=seeds[:3], **MAACO_DEFAULT)
    assert b.max_cells == default_max_cells(48, 48) < 1174
    assert b.solve() == want[:3]
    assert b.max_cells == 48 * 48                                           # the wave was repeated
    # the repeated wave is followed by waves with the default capacity: they must not take over its buffers
    seen = []

    class Recording(batch.MAACOBatch):
        def __init__(self, grids, *args, reuse=None, **kw):
            super().__init__(grids, *args, reuse=reuse, **kw)
            seen.append((self.n_maps, self.max_cells, reuse is not None and any(
                getattr(self, n).data_ptr() == getattr(reuse, n).data_ptr() for n in ("_tau", "_moves", "_best_cells"))))

    monkeypatch.setattr(batch, "MAACOBatch", Recording)
    res = solve_maaco_batch([grids[1], grids[0]] + grids[2:], N, K, MAACO_DEFAULT, seeds=[12, 11, 13, 14, 15], wave=2)
    assert seen == [(2, 1024, False), (2, 48 * 48, False),                  # the serpentine's wave, then its repeat
                    (2, 1024, False), (1, 1024, False)]
    assert [r[1:] for r in res] == [want[1], want[0]] + want[2:]
    with pytest.raises(MppError, match="outgrew max_cells=1024"):
        MAACOBatch(np.stack(grids[:3]), N, K, seeds=seeds[:3], max_cells=1024, **MAACO_DEFAULT).solve()


# ---- MPA -------------------------------------------------------------------------------------------------------------

def _mpa_solo(grid, N, K, seed, **params):
    """What MPA returns and stores for one map: (path, length, turns, safety, diag, fitness, convergence_curve)."""
    from maaco_path_planing_b200.mpa import MPA
    s = MPA(grid, num_predators=N, num_iterations=K, rng_seed=seed, verbose=False, **params)
    return tuple(s.solve_path_planning()) + (s.convergence_curve_data,)


def _mpa_oracle(grid, N, K, seed, p):
    from py_solvers import MpaOracle
    return MpaOracle(grid, N, K, p["FADs_rate"], p["P_const"], p["levy_beta"], p["turn_penalty_factor"],
                     p["safety_penalty_factor"], p["min_safe_distance"], p["diagonal_obstacle_penalty"], seed)


@pytest.mark.gpu
@pytest.mark.parametrize("beta,oracle_maps", [(2.0, (0, 3)), (1.5, (3,))])
def test_mpa_config5_wave(beta, oracle_maps):
    """MPABatch at the config-5 MPA shape: 256x256 maps, 1024 predators, 6 iterations (two of each phase).  Every map
    == solo MPA; some == the oracle; the same wave with 8 search warps per map and as one-map batches is identical."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MPABatch
    p = dict(MPA_PARAMS, levy_beta=beta)
    M, N, K = 4, 1024, 6
    grids = np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(M)])
    seeds = list(range(M))
    b = MPABatch(grids, N, K, seeds=seeds, **p)
    assert b.warps_per_map > 8
    res = b.solve()
    for i in range(M):
        assert res[i] == _mpa_solo(grids[i], N, K, seeds[i], **p), i
    for i in oracle_maps:
        o = _mpa_oracle(grids[i], N, K, seeds[i], p)
        opath, ost = o.solve()
        assert res[i][6] == o.curve and cells_of(res[i][0], 256) == list(opath) and res[i][5] == ost[4], i
    assert MPABatch(grids, N, K, seeds=seeds, warps_per_map=8, **p).solve() == res
    assert [MPABatch(grids[i:i + 1], N, K, seeds=seeds[i:i + 1], **p).solve()[0] for i in range(M)] == res


@pytest.mark.gpu
def test_mpa_wave_with_mixed_endpoints():
    """Unlike MAACO, one MPA wave may mix start / target cells (every search reads its own map's); one map's start is
    walled in, so its population is the reference's fallback path."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MPABatch
    ends = [((0, 0), (63, 63)), ((0, 63), (63, 0)), ((63, 63), (0, 0)), ((10, 50), (40, 5))]
    grids = [with_endpoints(blocks_map(64, 0.20, seed=640 + i), *ends[i]) for i in range(4)] + \
            [walled_in(blocks_map(64, 0.20, seed=644))]
    seeds = [21, 22, 23, 24, 25]
    N, K = 256, 6
    res = MPABatch(np.stack(grids), N, K, seeds=seeds, **MPA_PARAMS).solve()
    for i, g in enumerate(grids):
        assert res[i] == _mpa_solo(g, N, K, seeds[i], **MPA_PARAMS), i
    for i in range(len(grids)):
        o = _mpa_oracle(grids[i], N, K, seeds[i], MPA_PARAMS)
        opath, ost = o.solve()
        assert res[i][6] == o.curve and cells_of(res[i][0], 64) == list(opath) and res[i][5] == ost[4], i
    assert all(res[i][0][0] == ends[i][0] and res[i][0][-1] == ends[i][1] for i in range(4))


@pytest.mark.gpu
def test_mpa_config2_full_population_vs_oracle():
    """BASELINE config 2: MPA on bench.py's 100x100 map with 1024 predators, 12 iterations, against the oracle's mirror
    of the solve loop -- the curve, the best path and fitness, and every predator's final path.  The same map as a
    one-map MPABatch returns the same."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MPABatch
    from maaco_path_planing_b200.mpa import MPA
    g = blocks_map(100, 0.20, seed=2000)
    N, K, seed = 1024, 12, 2
    s = MPA(g, num_predators=N, num_iterations=K, rng_seed=seed, verbose=False, **MPA_PARAMS)
    res = s.solve_path_planning()
    o = _mpa_oracle(g, N, K, seed, MPA_PARAMS)
    opath, ost = o.solve()
    assert s.convergence_curve_data == o.curve
    assert cells_of(res[0], 100) == list(opath) and res[5] == ost[4]
    cells, ncell = s._pop["cells"].cpu().numpy(), s._pop["ncell"].cpu().numpy()
    for i, ind in enumerate(o.pop):
        assert np.array_equal(cells[i, :ncell[i]], np.array(ind["path"], np.int32)), f"predator {i}"
    assert MPABatch(g[None], N, K, seeds=[seed], **MPA_PARAMS).solve()[0] == tuple(res) + (s.convergence_curve_data,)
