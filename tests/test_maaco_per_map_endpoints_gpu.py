"""MAACOBatch(per_map_endpoints=True) and solve_maaco_batch(per_map_endpoints=True): waves whose maps have their own
start and target, one eta'**beta table per map (mpp_maaco_e01_host) and tau0 per map on the device
(mpp_maaco_tau0_maps).  Everything is compared bit for bit with solo MAACO and, on some maps, the C oracle."""
import numpy as np
import pytest

from conftest import MAACO_DEFAULT

INF = float("inf")
ORACLE_MAPS = (0, 1, 63, 64, 126, 127)


def with_endpoints(g, start, target):
    """`g` with its start and target moved to the given cells (their 2x2 corners cleared, like blocks_map's)."""
    g = g.copy()
    g[(g == 2) | (g == 3)] = 0
    for (r, c), v in ((start, 2), (target, 3)):
        r0, c0 = min(r, g.shape[0] - 2), min(c, g.shape[1] - 2)
        g[r0:r0 + 2, c0:c0 + 2] = 0
        g[r, c] = v
    return g


def moved(grids, seed):
    """The maps with start and target moved to seeded random free cells."""
    rng = np.random.default_rng(seed)
    out = np.array(grids, copy=True)
    for g in out:
        g[g >= 2] = 0
        s, t = rng.choice(np.flatnonzero(g.ravel() == 0), 2, replace=False)
        g.flat[s], g.flat[t] = 2, 3
    return out


def serpentine(n=48):
    """One-cell-wide corridor whose only path visits every free cell (1175 cells at n = 48)."""
    g = np.zeros((n, n), np.int64)
    for k, r in enumerate(range(1, n, 2)):
        g[r, :] = 1
        if r < n - 1:
            g[r, n - 1 if k % 2 == 0 else 0] = 0
    g[0, 0] = 2
    g[n - 2, 0 if (n // 2 - 1) % 2 else n - 1] = 3
    return g


def solo(grid, N, K, seed):
    from maaco_path_planing_b200 import MAACO
    return MAACO(grid, N, K, rng_seed=seed, verbose=False, **MAACO_DEFAULT)


def solo_solve(grid, N, K, seed):
    m = solo(grid, N, K, seed)
    path, length, turns = m.solve_path_planning()
    return path, length, turns, m.convergence_curve_data


def hard_pairs(R, Cc):
    """Endpoint pairs on one row / one column (orientation with fast_ok = 0), adjacent, corner to corner, diagonal."""
    return [((3, 5), (3, Cc - 4)), ((R - 2, Cc - 3), (R - 2, 1)), ((2, 40), (R - 3, 40)), ((R - 1, 9), (0, 9)),
            ((20, 20), (20, 21)), ((20, 20), (21, 21)), ((0, 0), (R - 1, Cc - 1)), ((R - 1, 0), (0, Cc - 1)),
            ((10, 12), (R - 10, Cc - 15)), ((R - 5, Cc - 7), (4, 6))]


def mixed_maps(R, Cc, n, seed):
    from maaco_path_planing_b200 import blocks_map
    base = [blocks_map(max(R, Cc), 0.20, seed=seed + i)[:R, :Cc] for i in range(n)]
    pairs = hard_pairs(R, Cc)
    out = [with_endpoints(g, *pairs[i]) for i, g in enumerate(base[:len(pairs)])]
    if n > len(pairs):
        out += list(moved(np.stack(base[len(pairs):]), seed))
    return np.stack(out)


@pytest.mark.gpu
def test_tables_per_map_from_host_and_device_grids():
    """Before any pass, map k's tau equals MAACO(grid_k).pheromone_matrix and its E01 row MAACO(grid_k)._E01."""
    import torch
    from maaco_path_planing_b200.batch import MAACOBatch
    grids = mixed_maps(64, 96, 40, 9600)
    assert len({(int(np.argmax(g == 2)), int(np.argmax(g == 3))) for g in grids}) == 40
    want = [solo(g, 8, 2, 1) for g in grids]
    for src in (grids, torch.from_numpy(grids).cuda()):
        b = MAACOBatch(src, 8, 2, seeds=range(40), per_map_endpoints=True, **MAACO_DEFAULT)
        assert b.per_map_tables and tuple(b._E01.shape) == (40, 2 * 64 * 96)
        tau, e01 = b.pheromone(), b._E01.cpu().numpy()
        for k, m in enumerate(want):
            assert tau[k].tobytes() == m.pheromone_matrix.tobytes(), k
            assert e01[k].tobytes() == m._E01.cpu().numpy().tobytes(), k


@pytest.mark.gpu
def test_config5_wave_random_endpoints_vs_solo_and_oracle():
    """128 256x256 maps with random endpoints x 1024 ants in one per-map wave: passes 1-2 per ant and tau against solo
    MAACO for every map and the C oracle on six maps, then the solve."""
    import pyoracle as O
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    M, N, K = 128, 1024, 3
    grids = moved(np.stack([blocks_map(256, 0.20, seed=5000 + i) for i in range(M)]), 5000)
    seeds = list(range(M))
    b = MAACOBatch(grids, N, K, seeds=seeds, per_map_endpoints=True, **MAACO_DEFAULT)
    assert b.per_map_tables
    passes = []
    for it in (1, 2):
        b.run_iteration(it)
        passes.append(b.last_results() + (b.pheromone(),))
    res = b.solve()
    assert (passes[1][0] > 0).sum() > 1000                  # random endpoints are far apart: few tours arrive early
    for i in range(M):
        s = solo(grids[i], N, K, seeds[i])
        orc = O.MaacoOracle(grids[i], N, K, seed=seeds[i], threads=0, **MAACO_DEFAULT) if i in ORACLE_MAPS else None
        for it, (bnc, bln, btn, btau) in enumerate(passes, 1):
            s.run_iteration(it)
            snc, sln, stn = s.last_results()
            assert np.array_equal(bnc[i], snc) and np.array_equal(bln[i], sln) and np.array_equal(btn[i], stn), (i, it)
            assert np.array_equal(btau[i], s.pheromone_matrix), (i, it)
            if orc is not None:
                _, onc, oln, otn, _ = orc.iterate(it)
                assert np.array_equal(bnc[i], onc) and np.array_equal(bln[i], oln) and np.array_equal(btn[i], otn), (i, it)
                assert np.array_equal(btau[i].ravel(), orc.tau), (i, it)
        path, length, turns = s.solve_path_planning()
        assert res[i] == (path, length, turns, s.convergence_curve_data), i


@pytest.mark.gpu
def test_shared_endpoints_take_the_shared_table():
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    grids = np.stack([blocks_map(64, 0.20, seed=640 + i) for i in range(4)])
    N, K = 128, 3
    b = MAACOBatch(grids, N, K, seeds=[1, 2, 3, 4], per_map_endpoints=True, **MAACO_DEFAULT)
    d = MAACOBatch(grids, N, K, seeds=[1, 2, 3, 4], **MAACO_DEFAULT)
    assert not b.per_map_tables and tuple(b._E01.shape) == (2 * 64 * 64,) and b._colony.E01_stride == 0
    assert b.solve() == d.solve()


@pytest.mark.gpu
def test_hard_cases_in_one_wave():
    """A walled-in start, one-row / one-column pairs beside diagonal ones, and a ragged 100x150 shape with targets in the
    last tile row / column, each in one per-map wave."""
    from maaco_path_planing_b200.batch import MAACOBatch
    N, K = 128, 3
    grids = mixed_maps(64, 64, 10, 6400)
    grids[8] = with_endpoints(grids[8], (0, 0), (50, 40))
    grids[8][0, 1] = grids[8][1, 0] = grids[8][1, 1] = 1                    # walled in
    res = MAACOBatch(grids, N, K, seeds=range(10), per_map_endpoints=True, **MAACO_DEFAULT).solve()
    for k, g in enumerate(grids):
        assert res[k] == solo_solve(g, N, K, k), k
    assert res[8] == ([], INF, INF, [None] * K)
    assert all(r[0] for k, r in enumerate(res) if k != 8)
    pairs = [((3, 4), (98, 140)), ((97, 149), (2, 2)), ((50, 0), (99, 130)), ((10, 145), (99, 149)), ((99, 0), (0, 149))]
    grids = mixed_maps(100, 150, 5, 1500)
    grids = np.stack([with_endpoints(g, *p) for g, p in zip(grids, pairs)])
    res = MAACOBatch(grids, N, K, seeds=range(5), per_map_endpoints=True, **MAACO_DEFAULT).solve()
    for k, g in enumerate(grids):
        assert res[k] == solo_solve(g, N, K, k), k


@pytest.mark.gpu
def test_reuse_between_per_map_and_shared_waves():
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    N, K, M = 128, 3, 4
    waves = [mixed_maps(64, 64, M, 700 + 10 * w) for w in range(2)]
    shared = np.stack([blocks_map(64, 0.20, seed=790 + i) for i in range(M)])
    mk = lambda g, seeds, **kw: MAACOBatch(g, N, K, seeds=seeds, per_map_endpoints=True, **MAACO_DEFAULT, **kw)
    a = mk(waves[0], range(M))
    a.run_iteration(1)
    b = mk(waves[1], range(M, 2 * M), reuse=a)
    for name in ("_tau", "_E01", "_moves", "_best_cells", "_log"):
        assert getattr(b, name).data_ptr() == getattr(a, name).data_ptr(), name
    fresh = mk(waves[1], range(M, 2 * M))
    for it in range(1, K + 1):
        b.run_iteration(it)
        fresh.run_iteration(it)
        for x, y in zip(b.last_results(), fresh.last_results()):
            assert np.array_equal(x, y), it
        assert np.array_equal(b.pheromone(), fresh.pheromone()), it
    assert b.solve() == fresh.solve()
    s = mk(shared, range(M))
    assert not s.per_map_tables
    s.run_iteration(1)
    c = mk(waves[0], range(M), reuse=s)
    assert tuple(c._E01.shape) == (M, 2 * 64 * 64) and c._E01.data_ptr() != s._E01.data_ptr()
    res = c.solve()
    for k in range(M):
        assert res[k] == solo_solve(waves[0][k], N, K, k), k


@pytest.mark.gpu
def test_path_capacity_repeat_keeps_the_tables():
    from maaco_path_planing_b200 import MppError, blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch, default_max_cells
    grids = np.stack([serpentine(), with_endpoints(blocks_map(48, 0.20, seed=481), (0, 47), (47, 0)),
                      with_endpoints(blocks_map(48, 0.20, seed=482), (20, 3), (30, 44))])
    N, K, seeds = 32, 3, [11, 12, 13]
    want = [solo_solve(g, N, K, s) for g, s in zip(grids, seeds)]
    assert len(want[0][0]) == 1175
    b = MAACOBatch(grids, N, K, seeds=seeds, per_map_endpoints=True, **MAACO_DEFAULT)
    assert b.per_map_tables and b.max_cells == default_max_cells(48, 48)
    e01 = b._E01.data_ptr()
    assert b.solve() == want
    assert b.max_cells == 48 * 48 and b.per_map_tables and b._E01.data_ptr() == e01    # repeated on the same tables
    with pytest.raises(MppError, match="outgrew max_cells=1024"):
        MAACOBatch(grids, N, K, seeds=seeds, max_cells=1024, per_map_endpoints=True, **MAACO_DEFAULT).solve()


def _three_endpoint_maps():
    from maaco_path_planing_b200 import blocks_map
    ends = [((0, 0), (63, 63)), ((0, 63), (63, 0)), ((63, 63), (0, 0))]
    labels = [0, 1, 2] * 4 + [0, 1, 0, 1, 0, 1, 1]
    return [with_endpoints(blocks_map(64, 0.20, seed=700 + i), *ends[e]) for i, e in enumerate(labels)]


@pytest.mark.gpu
def test_sweep_waves_by_shape_in_index_order(monkeypatch):
    import torch
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch
    grids = _three_endpoint_maps()
    seeds = [40 + i for i in range(len(grids))]
    seen = []

    class Recording(batch.MAACOBatch):
        def __init__(self, grids, *args, reuse=None, **kw):
            super().__init__(grids, *args, reuse=reuse, **kw)
            seen.append((self.n_maps, self.per_map_tables, tuple(self._map_set.start),
                         reuse is not None and self._moves.data_ptr() == reuse._moves.data_ptr()))

    monkeypatch.setattr(batch, "MAACOBatch", Recording)
    N, K = 128, 3
    res = solve_maaco_batch(grids, N, K, MAACO_DEFAULT, seeds=seeds, wave=3, per_map_endpoints=True)
    starts = [int(np.argmax(g.ravel() == 2)) for g in grids]
    assert [s[0] for s in seen] == [3] * 6 + [1]
    assert [s[2] for s in seen] == [tuple(starts[w:w + 3]) for w in range(0, 19, 3)]
    assert [s[3] for s in seen] == [False] + [True] * 5 + [False]
    assert all(s[1] for s in seen[:6])
    want = [solo_solve(g, N, K, s) for g, s in zip(grids, seeds)]
    assert [r[0] for r in res] == list(range(len(grids))) and [r[1:] for r in res] == want
    # device grids: one 3-D tensor and a list of 2-D tensors
    dev = torch.from_numpy(np.stack(grids)).cuda()
    assert solve_maaco_batch(dev, N, K, MAACO_DEFAULT, seeds=seeds, wave=3, per_map_endpoints=True) == res
    assert solve_maaco_batch(list(dev), N, K, MAACO_DEFAULT, seeds=seeds, wave=3, per_map_endpoints=True) == res
    # two shapes interleaved: waves per shape, in index order
    from maaco_path_planing_b200 import blocks_map
    two = [g if i % 2 else with_endpoints(blocks_map(80, 0.2, seed=800 + i)[:48], (0, 5), (47, 70))
           for i, g in enumerate(grids[:7])]
    two[4] = with_endpoints(two[4], (47, 0), (0, 79))
    seen.clear()
    res2 = solve_maaco_batch(two, N, K, MAACO_DEFAULT, seeds=seeds[:7], wave=2, per_map_endpoints=True)
    assert [s[0] for s in seen] == [2, 2, 2, 1]
    assert [r[1:] for r in res2] == [solo_solve(g, N, K, s) for g, s in zip(two, seeds[:7])]
    # seeds=None runs
    res3 = solve_maaco_batch(grids[:4], N, K, MAACO_DEFAULT, wave=3, per_map_endpoints=True)
    assert [r[0] for r in res3] == [0, 1, 2, 3] and all(r[1] for r in res3)


@pytest.mark.gpu
def test_sweep_missing_endpoint_raises_before_device_work(monkeypatch):
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch
    grids = _three_endpoint_maps()[:7]

    class Never(batch.MAACOBatch):
        def __init__(self, *a, **kw):
            raise AssertionError("a wave ran before the endpoint check")

    monkeypatch.setattr(batch, "MAACOBatch", Never)
    for v, msg in ((2, "MAACO: Start node not found."), (3, "MAACO: Target node not found.")):
        bad = [g.copy() for g in grids]
        bad[5][bad[5] == v] = 0
        with pytest.raises(ValueError, match=msg):
            solve_maaco_batch(bad, 64, 2, MAACO_DEFAULT, wave=3, per_map_endpoints=True)


@pytest.mark.gpu
def test_side_stream_equals_default_stream():
    import torch
    from maaco_path_planing_b200.batch import MAACOBatch
    grids = mixed_maps(64, 64, 6, 6460)
    N, K = 256, 3
    want = MAACOBatch(grids, N, K, seeds=range(6), per_map_endpoints=True, **MAACO_DEFAULT).solve()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        got = MAACOBatch(grids, N, K, seeds=range(6), per_map_endpoints=True, **MAACO_DEFAULT).solve()
    assert got == want
