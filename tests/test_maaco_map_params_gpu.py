"""MAACOBatch(map_params=...) and solve_maaco_batch(map_params=...): waves whose maps each have their own colony
parameters, run by the per-map instantiations of the table and pass kernels (mpp_maaco_tau0_maps_p,
mpp_maaco_e01_maps_p, mpp_maaco_pass_maps).  Map k must give what solo MAACO gives with map k's parameters and seed,
bit for bit, alpha != 1 included; on alpha == 1 maps also what the C oracle gives."""
import numpy as np
import pytest

from conftest import MAACO_DEFAULT
from test_maaco_per_map_endpoints_gpu import mixed_maps, serpentine, with_endpoints

INF = float("inf")


def param_sets(n, seed, alphas=(1.0, 0.5, 2.0)):
    """n seeded parameter sets that vary every key; alpha cycles through `alphas`."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        out.append(dict(alpha=alphas[i % len(alphas)], beta=float(rng.uniform(5.0, 8.0)), rho=float(rng.uniform(0.05, 0.3)),
                        Q=float(rng.uniform(1.0, 5.0)), a_turn_coef=float(rng.uniform(0.5, 2.0)),
                        wh_max=float(rng.uniform(0.8, 0.95)), wh_min=float(rng.uniform(0.1, 0.3)),
                        k_h_adaptive=float(rng.uniform(0.5, 1.5)), q0_initial=float(rng.uniform(0.2, 0.9)),
                        C0_initial_pheromone=float(rng.uniform(0.05, 0.5))))
    return out


def solo(grid, N, K, seed, params):
    from maaco_path_planing_b200 import MAACO
    return MAACO(grid, N, K, rng_seed=seed, verbose=False, **params)


def solo_solve(grid, N, K, seed, params):
    m = solo(grid, N, K, seed, params)
    path, length, turns = m.solve_path_planning()
    return path, length, turns, m.convergence_curve_data


@pytest.mark.gpu
@pytest.mark.parametrize("host_e01", [False, True])
def test_tables_per_map_params(monkeypatch, host_e01):
    """16 parameter sets on one 64x96 map, then 16 maps with their own endpoints: before any pass, map k's tau and E01
    are MAACO(grid_k, **params_k)'s, byte for byte, from host and device grids (host_e01: the tables built by
    mpp_maaco_e01_host, once per distinct set, as where the device's exp / pow do not match the host libm)."""
    import torch
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import MAACOBatch
    if host_e01:
        monkeypatch.setattr(batch, "_DEVICE_E01", False)
    ps = param_sets(16, 1600)
    ps[5] = dict(ps[4], alpha=3.0, rho=0.5)                   # two maps share their table parameters
    one = mixed_maps(64, 96, 1, 9601)[0]
    for grids, per_map_endpoints in ((np.stack([one] * 16), False), (mixed_maps(64, 96, 16, 9602), True)):
        want = [solo(g, 8, 2, 1, p) for g, p in zip(grids, ps)]
        for src in (grids, torch.from_numpy(grids).cuda()):
            b = MAACOBatch(src, 8, 2, seeds=range(16), per_map_endpoints=per_map_endpoints, map_params=ps,
                           **MAACO_DEFAULT)
            assert b.per_map_tables and tuple(b._E01.shape) == (16, 2 * 64 * 96)
            assert b.map_params == ps
            tau, e01 = b.pheromone(), b._E01.cpu().numpy()
            for k, m in enumerate(want):
                assert tau[k].tobytes() == m.pheromone_matrix.tobytes(), k
                assert e01[k].tobytes() == m._E01.cpu().numpy().tobytes(), k


@pytest.mark.gpu
def test_sweep_wave_pass_by_pass_vs_solo_and_oracle():
    """64 parameter sets on 64 256x256 maps x 1024 ants in one wave, alpha 1 / 0.5 / 2 mixed: per-ant results and tau
    after each of 3 passes against solo MAACO with each map's parameters, and the C oracle on alpha == 1 maps."""
    import pyoracle as O
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    M, N, K = 64, 1024, 3
    grids = np.stack([blocks_map(256, 0.20, seed=6400 + i) for i in range(M)])
    ps = param_sets(M, 6400)
    seeds = [1000 + i for i in range(M)]
    b = MAACOBatch(grids, N, K, seeds=seeds, map_params=ps, **MAACO_DEFAULT)
    assert b.per_map_tables
    passes = []
    for it in range(1, K + 1):
        b.run_iteration(it)
        passes.append(b.last_results() + (b.pheromone(),))
    res = b.solve()
    assert (passes[-1][0] > 0).sum() > 1000
    oracle_maps = (0, 3, 63)
    assert all(ps[i]["alpha"] == 1.0 for i in oracle_maps)
    for i in range(M):
        s = solo(grids[i], N, K, seeds[i], ps[i])
        orc = O.MaacoOracle(grids[i], N, K, seed=seeds[i], threads=0, **ps[i]) if i in oracle_maps else None
        for it, (bnc, bln, btn, btau) in enumerate(passes, 1):
            s.run_iteration(it)
            snc, sln, stn = s.last_results()
            assert np.array_equal(bnc[i], snc) and np.array_equal(bln[i], sln) and np.array_equal(btn[i], stn), (i, it)
            assert btau[i].tobytes() == s.pheromone_matrix.tobytes(), (i, it)
            if orc is not None:
                _, onc, oln, otn, _ = orc.iterate(it)
                assert np.array_equal(bnc[i], onc) and np.array_equal(bln[i], oln) and np.array_equal(btn[i], otn), (i, it)
                assert np.array_equal(btau[i].ravel(), orc.tau), (i, it)
        path, length, turns = s.solve_path_planning()
        assert res[i] == (path, length, turns, s.convergence_curve_data), i


@pytest.mark.gpu
def test_constructor_parameters_per_map_change_nothing():
    """map_params that give every map the constructor's parameters: the bytes of map_params=None, pass by pass."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    grids = np.stack([blocks_map(96, 0.20, seed=960 + i) for i in range(8)])
    N, K = 256, 4
    a = MAACOBatch(grids, N, K, seeds=range(8), **MAACO_DEFAULT)
    b = MAACOBatch(grids, N, K, seeds=range(8), map_params=[dict(MAACO_DEFAULT)] * 4 + [{}] * 4, **MAACO_DEFAULT)
    assert a.map_params is None and b.map_params == [{k: float(v) for k, v in MAACO_DEFAULT.items()}] * 8
    assert not b.per_map_tables and a._E01.cpu().numpy().tobytes() == b._E01.cpu().numpy().tobytes()
    assert a.pheromone().tobytes() == b.pheromone().tobytes()
    for it in range(1, K + 1):
        a.run_iteration(it)
        b.run_iteration(it)
        for x, y in zip(a.last_results(), b.last_results()):
            assert x.tobytes() == y.tobytes(), it
        assert a.pheromone().tobytes() == b.pheromone().tobytes(), it
    assert a.solve() == b.solve()
    assert a._log.cpu().numpy().tobytes() == b._log.cpu().numpy().tobytes()


@pytest.mark.gpu
def test_path_capacity_repeat_keeps_map_params():
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch, default_max_cells
    grids = np.stack([serpentine(), with_endpoints(blocks_map(48, 0.20, seed=481), (0, 47), (47, 0)),
                      with_endpoints(blocks_map(48, 0.20, seed=482), (20, 3), (30, 44))])
    N, K, seeds = 32, 3, [11, 12, 13]
    ps = [dict(alpha=2.0, rho=0.2), dict(beta=6.0, q0_initial=0.8), dict(alpha=0.5, Q=4.0, C0_initial_pheromone=0.3)]
    full = [{**MAACO_DEFAULT, **p} for p in ps]
    want = [solo_solve(g, N, K, s, p) for g, s, p in zip(grids, seeds, full)]
    assert len(want[0][0]) == 1175
    b = MAACOBatch(grids, N, K, seeds=seeds, per_map_endpoints=True, map_params=ps, **MAACO_DEFAULT)
    assert b.per_map_tables and b.max_cells == default_max_cells(48, 48)
    e01 = b._E01.data_ptr()
    assert b.solve() == want
    assert b.max_cells == 48 * 48 and b._E01.data_ptr() == e01                  # repeated on the same tables
    assert b.map_params == [{k: float(v) for k, v in p.items()} for p in full]


@pytest.mark.gpu
def test_reuse_between_map_params_and_default_waves():
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    N, K, M = 128, 3, 4
    grids = [np.stack([blocks_map(64, 0.20, seed=1300 + 10 * w + i) for i in range(M)]) for w in range(3)]
    ps = [param_sets(M, 130 + w) for w in range(3)]
    a = MAACOBatch(grids[0], N, K, seeds=range(M), map_params=ps[0], **MAACO_DEFAULT)
    a.run_iteration(1)
    d = MAACOBatch(grids[1], N, K, seeds=range(M), reuse=a, **MAACO_DEFAULT)          # a default wave: its own buffers
    assert d._moves.data_ptr() != a._moves.data_ptr() and d._key != a._key
    assert d.solve() == MAACOBatch(grids[1], N, K, seeds=range(M), **MAACO_DEFAULT).solve()
    b = MAACOBatch(grids[2], N, K, seeds=range(M, 2 * M), map_params=ps[2], reuse=a, **MAACO_DEFAULT)
    for name in ("_tau", "_E01", "_moves", "_best_cells", "_log"):
        assert getattr(b, name).data_ptr() == getattr(a, name).data_ptr(), name
    fresh = MAACOBatch(grids[2], N, K, seeds=range(M, 2 * M), map_params=ps[2], **MAACO_DEFAULT)
    for it in range(1, K + 1):
        b.run_iteration(it)
        fresh.run_iteration(it)
        for x, y in zip(b.last_results(), fresh.last_results()):
            assert np.array_equal(x, y), it
        assert np.array_equal(b.pheromone(), fresh.pheromone()), it
    res = b.solve()
    assert res == fresh.solve()
    for k in range(M):
        assert res[k] == solo_solve(grids[2][k], N, K, M + k, ps[2][k]), k
    c = MAACOBatch(grids[1], N, K, seeds=range(M), reuse=b, **MAACO_DEFAULT)          # and back to a default wave
    assert c.solve() == d.solve()


def _sweep_maps():
    """Two shapes interleaved; 64x64 maps with three endpoint pairs, 48x80 maps with two."""
    from maaco_path_planing_b200 import blocks_map
    ends = [((0, 0), (63, 63)), ((0, 63), (63, 0)), ((63, 63), (0, 0))]
    out = []
    for i in range(13):
        if i % 3 == 2:
            pair = ((0, 5), (47, 70)) if i % 2 else ((47, 0), (0, 79))
            out.append(with_endpoints(blocks_map(80, 0.2, seed=820 + i)[:48], *pair))
        else:
            out.append(with_endpoints(blocks_map(64, 0.20, seed=720 + i), *ends[i % 3]))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("per_map_endpoints", [False, True])
def test_sweep_with_map_params(monkeypatch, per_map_endpoints):
    import torch
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch
    grids = _sweep_maps()
    seeds = [50 + i for i in range(len(grids))]
    ps = param_sets(len(grids), 1313)
    seen = []

    class Recording(batch.MAACOBatch):
        def __init__(self, grids, *args, **kw):
            super().__init__(grids, *args, **kw)
            seen.append(self.n_maps)

    monkeypatch.setattr(batch, "MAACOBatch", Recording)
    N, K = 128, 3
    res = solve_maaco_batch(grids, N, K, MAACO_DEFAULT, seeds=seeds, wave=3, per_map_endpoints=per_map_endpoints,
                            map_params=ps)
    plain = list(seen)
    seen.clear()
    solve_maaco_batch(grids, N, K, MAACO_DEFAULT, seeds=seeds, wave=3, per_map_endpoints=per_map_endpoints)
    assert seen == plain                                                       # parameters never split waves
    want = [solo_solve(g, N, K, s, p) for g, s, p in zip(grids, seeds, ps)]
    assert [r[0] for r in res] == list(range(len(grids))) and [r[1:] for r in res] == want
    assert solve_maaco_batch([torch.from_numpy(g).cuda() for g in grids], N, K, MAACO_DEFAULT, seeds=seeds, wave=3,
                             per_map_endpoints=per_map_endpoints, map_params=ps) == res
    same = [g for g in grids if g.shape == (64, 64)]
    idx = [i for i, g in enumerate(grids) if g.shape == (64, 64)]
    got = solve_maaco_batch(torch.from_numpy(np.stack(same)).cuda(), N, K, MAACO_DEFAULT, seeds=[seeds[i] for i in idx],
                            wave=4, per_map_endpoints=per_map_endpoints, map_params=[ps[i] for i in idx])
    assert [r[1:] for r in got] == [want[i] for i in idx]


@pytest.mark.gpu
def test_sweep_bad_map_params_raise_before_any_wave(monkeypatch):
    import torch
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch
    grids = _sweep_maps()[:5]

    class Never(batch.MAACOBatch):
        def __init__(self, *a, **kw):
            raise AssertionError("a wave ran before map_params were checked")

    monkeypatch.setattr(batch, "MAACOBatch", Never)
    for src in (grids, torch.from_numpy(np.stack([g for g in grids if g.shape == (64, 64)])).cuda()):
        n = len(src)
        for mp, match in (([{}] * (n - 1), "entries for"), ([{}] * (n - 1) + [{"alpha2": 1.0}], "unknown parameter"),
                          ([{"num_iterations": 4}] + [{}] * (n - 1), "num_iterations")):
            with pytest.raises(ValueError, match=match):
                solve_maaco_batch(src, 64, 2, MAACO_DEFAULT, wave=3, per_map_endpoints=True, map_params=mp)


@pytest.mark.gpu
def test_batch_bad_map_params_raise():
    from maaco_path_planing_b200 import MppError, blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    grids = np.stack([blocks_map(32, 0.2, seed=i) for i in range(3)])
    for mp, match in (([{}] * 2, "2 entries for 3 maps"), ([{}, {"rho2": 0.1}, {}], "unknown parameter"),
                      ([{}, {}, {"num_ants": 4}], "num_ants")):
        with pytest.raises(ValueError, match=match):
            MAACOBatch(grids, 16, 2, seeds=range(3), map_params=mp, **MAACO_DEFAULT)
    moved = np.stack([grids[0], with_endpoints(grids[1], (0, 31), (31, 0)), grids[2]])
    with pytest.raises(MppError, match="must share start and target"):
        MAACOBatch(moved, 16, 2, seeds=range(3), map_params=[{}] * 3, **MAACO_DEFAULT)


@pytest.mark.gpu
def test_side_stream_equals_default_stream():
    import torch
    from maaco_path_planing_b200.batch import MAACOBatch
    grids = mixed_maps(64, 64, 6, 6461)
    ps = param_sets(6, 6461)
    N, K = 256, 3
    want = MAACOBatch(grids, N, K, seeds=range(6), per_map_endpoints=True, map_params=ps, **MAACO_DEFAULT).solve()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        got = MAACOBatch(grids, N, K, seeds=range(6), per_map_endpoints=True, map_params=ps, **MAACO_DEFAULT).solve()
    assert got == want
    for k in range(6):
        assert want[k] == solo_solve(grids[k], N, K, k, ps[k]), k
