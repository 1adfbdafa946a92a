"""MAACOBatch(map_sizes=...) and solve_maaco_batch(map_sizes=...): waves whose maps each have their own colony size and
pass count inside buffers sized for the wave's largest (mpp_maaco_pass_maps_sized).  Map k must give what solo
MAACO(grid_k, num_ants_k, num_iterations_k, ...) gives with map k's parameters and seed, bit for bit: per-ant records
and tau after every pass, and the solve's result."""
import ctypes as C

import numpy as np
import pytest

from conftest import MAACO_DEFAULT
from test_maaco_map_params_gpu import _sweep_maps, param_sets
from test_maaco_per_map_endpoints_gpu import mixed_maps, serpentine, with_endpoints

INF = float("inf")
ANTS = (1, 2, 31, 32, 33, 100, 255, 256, 1000, 1024)
PASSES = (0, 1, 2, 3, 5)


def mixed_sizes(n, seed):
    """n sizes that cover every value of ANTS and PASSES, in seeded combinations."""
    rng = np.random.default_rng(seed)
    a = [ANTS[i % len(ANTS)] for i in range(n)]
    k = [PASSES[i % len(PASSES)] for i in range(n)]
    rng.shuffle(a)
    rng.shuffle(k)
    return [{"num_ants": int(x), "num_iterations": int(y)} for x, y in zip(a, k)]


def solo(grid, s, seed, params=None):
    from maaco_path_planing_b200 import MAACO
    return MAACO(grid, s["num_ants"], s["num_iterations"], rng_seed=seed, verbose=False,
                 **{**MAACO_DEFAULT, **(params or {})})


def solo_solve(grid, s, seed, params=None):
    m = solo(grid, s, seed, params)
    path, length, turns = m.solve_path_planning()
    return path, length, turns, m.convergence_curve_data


def failed(nc, ln, tn):
    return (nc == 0).all() and np.isinf(ln).all() and (ln > 0).all() and (tn == -1).all()


def passes_of(b):
    """Runs every pass of `b`; (n_cells, length, turns, tau) after each."""
    out = []
    for it in range(1, b._passes + 1):
        b.run_iteration(it)
        out.append(b.last_results() + (b.pheromone(),))
    return out


def check_against_solo(grids, sizes, seeds, params, passes, res, tau_init, oracle_maps=()):
    import pyoracle as O
    for i, s in enumerate(sizes):
        n, K = s["num_ants"], s["num_iterations"]
        m = solo(grids[i], s, seeds[i], params[i] if params else None)
        assert tau_init[i].tobytes() == m.pheromone_matrix.tobytes(), i
        orc = O.MaacoOracle(grids[i], n, K, seed=seeds[i], threads=0, **MAACO_DEFAULT) if i in oracle_maps else None
        tau = tau_init[i]
        for it, (bnc, bln, btn, btau) in enumerate(passes, 1):
            if it <= K:
                m.run_iteration(it)
                snc, sln, stn = m.last_results()
                assert np.array_equal(bnc[i, :n], snc) and np.array_equal(bln[i, :n], sln), (i, it)
                assert np.array_equal(btn[i, :n], stn), (i, it)
                tau = m.pheromone_matrix
                if orc is not None:
                    _, onc, oln, otn, _ = orc.iterate(it)
                    assert np.array_equal(snc, onc) and np.array_equal(sln, oln) and np.array_equal(stn, otn), (i, it)
                    assert np.array_equal(tau.ravel(), orc.tau), (i, it)
            assert failed(bnc[i, n:], bln[i, n:], btn[i, n:]), (i, it)       # outside the colony
            if K == 0:
                assert failed(bnc[i], bln[i], btn[i]), (i, it)                  # never ran a pass
            assert btau[i].tobytes() == tau.tobytes(), (i, it)                  # frozen after the map's last pass
        path, length, turns = m.solve_path_planning()
        assert res[i] == (path, length, turns, m.convergence_curve_data), i
        assert len(res[i][3]) == K
        if K == 0:
            assert res[i] == ([], INF, INF, [])


@pytest.mark.gpu
def test_mixed_sizes_wave_pass_by_pass_vs_solo_and_oracle():
    """64 config-5 maps (256 x 256) with colonies of 1..1024 ants and 0..5 passes in one wave."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    M = 64
    grids = np.stack([blocks_map(256, 0.20, seed=7000 + i) for i in range(M)])
    sizes = mixed_sizes(M, 64)
    seeds = [3000 + i for i in range(M)]
    b = MAACOBatch(grids, 16, 2, seeds=seeds, map_sizes=sizes, **MAACO_DEFAULT)
    assert b.map_sizes == sizes and b._ants == 1024 and b._passes == 5 and tuple(b._log.shape) == (M, 5, 4)
    assert b.map_params == [{k: float(v) for k, v in MAACO_DEFAULT.items()}] * M
    assert failed(*b.last_results()) and b.last_results()[0].shape == (M, 1024)
    tau_init = b.pheromone()
    passes = passes_of(b)
    res = b.solve()
    assert sum(r[0] != [] for r in res) > 20
    oracle_maps = [i for i, s in enumerate(sizes) if s["num_iterations"] >= 2][:3]
    check_against_solo(grids, sizes, seeds, None, passes, res, tau_init, oracle_maps)


@pytest.mark.gpu
def test_sizes_with_map_params_and_per_map_endpoints():
    import torch
    from maaco_path_planing_b200.batch import MAACOBatch
    M = 12
    grids = mixed_maps(64, 64, M, 1212)
    ps = param_sets(M, 1212)
    sizes = [dict(s, num_ants=s["num_ants"] // 4 + 1) for s in mixed_sizes(M, 12)]
    seeds = [90 + i for i in range(M)]
    res = None
    for src in (grids, torch.from_numpy(grids).cuda()):
        b = MAACOBatch(src, 64, 3, seeds=seeds, per_map_endpoints=True, map_params=ps, map_sizes=sizes,
                       **MAACO_DEFAULT)
        assert b.per_map_tables
        tau_init = b.pheromone()
        passes = passes_of(b)
        got = b.solve()
        if res is None:
            res = got
            check_against_solo(grids, sizes, seeds, [{**MAACO_DEFAULT, **p} for p in ps], passes, got, tau_init)
        assert got == res


@pytest.mark.gpu
def test_constructor_sizes_change_nothing():
    """map_sizes that give every map the constructor's sizes: the bytes of the map_params wave and the default wave."""
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    M, N, K = 8, 200, 4
    grids = np.stack([blocks_map(96, 0.20, seed=960 + i) for i in range(M)])
    a = MAACOBatch(grids, N, K, seeds=range(M), **MAACO_DEFAULT)
    p = MAACOBatch(grids, N, K, seeds=range(M), map_params=[{}] * M, **MAACO_DEFAULT)
    s = MAACOBatch(grids, N, K, seeds=range(M), map_sizes=[{}] * 3 + [{"num_ants": N, "num_iterations": K}] * 5,
                   **MAACO_DEFAULT)
    assert s.map_sizes == [{"num_ants": N, "num_iterations": K}] * M and s.map_params == p.map_params
    for x in (p, s):
        assert x.pheromone().tobytes() == a.pheromone().tobytes()
    for it in range(1, K + 1):
        for x in (a, p, s):
            x.run_iteration(it)
        want = a.last_results()
        for x in (p, s):
            assert all(u.tobytes() == v.tobytes() for u, v in zip(x.last_results(), want)), it
            assert x.pheromone().tobytes() == a.pheromone().tobytes(), it
    res = a.solve()
    for x in (p, s):
        assert x.solve() == res
        assert x._log.cpu().numpy().tobytes() == a._log.cpu().numpy().tobytes()


@pytest.mark.gpu
def test_ants_per_warp_forms_agree():
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    M = 10
    grids = np.stack([blocks_map(128, 0.20, seed=1280 + i) for i in range(M)])
    sizes = mixed_sizes(M, 10)
    want = None
    for apw in (1, 2, 4, 8, 16, 32):
        b = MAACOBatch(grids, 8, 2, seeds=range(M), map_sizes=sizes, ants_per_warp=apw, **MAACO_DEFAULT)
        got = [x.tobytes() for p in passes_of(b) for x in p] + [b.solve(), b.total_steps()]
        if want is None:
            want = got
        assert got == want, apw


@pytest.mark.gpu
def test_repeat_reuse_and_steps():
    from maaco_path_planing_b200 import blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch, default_max_cells
    grids = np.stack([serpentine(), with_endpoints(blocks_map(48, 0.20, seed=481), (0, 47), (47, 0)),
                      with_endpoints(blocks_map(48, 0.20, seed=482), (20, 3), (30, 44)), serpentine()])
    sizes = [{"num_ants": 32, "num_iterations": 3}, {"num_ants": 5, "num_iterations": 1},
             {"num_ants": 17, "num_iterations": 0}, {"num_ants": 1, "num_iterations": 2}]
    seeds = [11, 12, 13, 14]
    want = [solo_solve(g, s, sd) for g, s, sd in zip(grids, sizes, seeds)]
    assert len(want[0][0]) == 1175
    b = MAACOBatch(grids, 8, 8, seeds=seeds, per_map_endpoints=True, map_sizes=sizes, **MAACO_DEFAULT)
    assert b.max_cells == default_max_cells(48, 48)
    assert b.solve() == want
    assert b.max_cells == 48 * 48 and b.map_sizes == sizes                     # repeated with the same sizes

    M = 6
    waves = [np.stack([blocks_map(64, 0.20, seed=1400 + 10 * w + i) for i in range(M)]) for w in range(3)]
    mixes = [[{"num_ants": n, "num_iterations": k} for n, k in zip(ns, ks)]
             for ns, ks in (([256, 3, 64, 100, 1, 33], [4, 0, 2, 4, 1, 3]), ([1, 256, 256, 7, 40, 90], [1, 2, 4, 0, 3, 4]),
                            ([256, 2, 2, 2, 2, 2], [4, 4, 4, 4, 4, 4]))]
    prev = None
    for w in range(3):
        b = MAACOBatch(waves[w], 16, 2, seeds=range(w, w + M), map_sizes=mixes[w], reuse=prev, **MAACO_DEFAULT)
        if prev is not None:
            assert b._key == prev._key and b._slabs.data_ptr() == prev._slabs.data_ptr()
        fresh = MAACOBatch(waves[w], 16, 2, seeds=range(w, w + M), map_sizes=mixes[w], **MAACO_DEFAULT)
        for x, y in zip(passes_of(b), passes_of(fresh)):
            assert all(u.tobytes() == v.tobytes() for u, v in zip(x, y)), w
        res = b.solve()
        assert res == fresh.solve()
        steps = 0
        for k in range(M):
            m = solo(waves[w][k], mixes[w][k], w + k)
            path, length, turns = m.solve_path_planning()
            assert res[k] == (path, length, turns, m.convergence_curve_data), (w, k)
            steps += m.total_steps()
        assert b.total_steps() == fresh.total_steps() == steps, w
        prev = b


@pytest.mark.gpu
@pytest.mark.parametrize("per_map_endpoints", [False, True])
def test_sweep_with_map_sizes(monkeypatch, per_map_endpoints):
    import torch
    from maaco_path_planing_b200 import batch
    from maaco_path_planing_b200.batch import solve_maaco_batch
    grids = _sweep_maps()
    seeds = [50 + i for i in range(len(grids))]
    sizes = [dict(s, num_ants=s["num_ants"] // 8 + 1) for s in mixed_sizes(len(grids), 1313)]
    seen = []

    class Recording(batch.MAACOBatch):
        def __init__(self, grids, *args, **kw):
            super().__init__(grids, *args, **kw)
            seen.append(self.n_maps)

    monkeypatch.setattr(batch, "MAACOBatch", Recording)
    res = solve_maaco_batch(grids, 64, 3, MAACO_DEFAULT, seeds=seeds, wave=3, per_map_endpoints=per_map_endpoints,
                            map_sizes=sizes)
    plain = list(seen)
    seen.clear()
    solve_maaco_batch(grids, 64, 3, MAACO_DEFAULT, seeds=seeds, wave=3, per_map_endpoints=per_map_endpoints)
    assert seen == plain                                                       # sizes never split waves
    want = [solo_solve(g, s, sd) for g, s, sd in zip(grids, sizes, seeds)]
    assert [r[0] for r in res] == list(range(len(grids))) and [r[1:] for r in res] == want
    assert solve_maaco_batch([torch.from_numpy(g).cuda() for g in grids], 64, 3, MAACO_DEFAULT, seeds=seeds, wave=3,
                             per_map_endpoints=per_map_endpoints, map_sizes=sizes) == res
    idx = [i for i, g in enumerate(grids) if g.shape == (64, 64)]
    got = solve_maaco_batch(torch.from_numpy(np.stack([grids[i] for i in idx])).cuda(), 64, 3, MAACO_DEFAULT,
                            seeds=[seeds[i] for i in idx], wave=4, per_map_endpoints=per_map_endpoints,
                            map_sizes=[sizes[i] for i in idx])
    assert [r[1:] for r in got] == [want[i] for i in idx]


@pytest.mark.gpu
def test_abi_clamps_sizes():
    """mpp_maaco_pass_maps_sized with out-of-range sizes, as the header documents them: a colony above the capacity runs
    the capacity, a colony of 0 constructs no tour and deposits nothing, a negative pass count takes part in no pass."""
    import torch
    from maaco_path_planing_b200 import _lib, blocks_map
    from maaco_path_planing_b200.batch import MAACOBatch
    g = blocks_map(64, 0.20, seed=641)
    grids = np.stack([g] * 4)
    N, K, seeds = 96, 2, [5, 5, 5, 5]
    ref = MAACOBatch(grids, N, K, seeds=seeds, map_params=[{}] * 4, **MAACO_DEFAULT)   # every map at the capacity
    b = MAACOBatch(grids, N, K, seeds=seeds, map_sizes=[{}] * 4, **MAACO_DEFAULT)
    sizes = torch.tensor([[1 << 30, 1 << 30], [0, K], [N, -1], [-7, K]], dtype=torch.int32, device=b.device)
    tau0, state0 = b.pheromone(), b._state.cpu().numpy().tobytes()
    rho = MAACO_DEFAULT["rho"]
    tau_empty = tau0.copy()
    L = _lib.lib()
    stream = C.c_void_p(torch.cuda.current_stream(b.device).cuda_stream)
    for it in range(1, K + 1):
        ref.run_iteration(it)
        _lib.check(L.mpp_maaco_pass_maps_sized(b._maps, C.byref(b._colony), _lib.ptr(b._params_dev), _lib.ptr(b._q0_dev),
                                               _lib.ptr(sizes), it, N, 0, stream), "mpp_maaco_pass_maps_sized")
        nc, ln, tn = b.last_results()
        rnc, rln, rtn = ref.last_results()
        tau, rtau = b.pheromone(), ref.pheromone()
        assert nc[0].tobytes() == rnc[0].tobytes() and ln[0].tobytes() == rln[0].tobytes(), it
        assert tn[0].tobytes() == rtn[0].tobytes() and tau[0].tobytes() == rtau[0].tobytes(), it
        # colony 0 (and a negative colony): no tours; tau evaporates and is clipped with no best length (MAACO.py:304-332)
        b_len = float(64 + 64)
        tmax = (1.0 / (1.0 - rho)) * (1.0 / b_len)
        tmin = tmax / (2.0 * 64)
        tau_empty = np.minimum(np.maximum(tau_empty * (1.0 - rho), tmin), tmax)
        tau_empty[grids == 1] = 1e-9
        for k in (1, 3):
            assert failed(nc[k], ln[k], tn[k]) and tau[k].tobytes() == tau_empty[k].tobytes(), (k, it)
        assert failed(nc[2], ln[2], tn[2]) and tau[2].tobytes() == tau0[2].tobytes(), it   # no pass at all
    st = b._state.cpu().numpy().tobytes()
    w = len(st) // 4
    assert st[2 * w:3 * w] == state0[2 * w:3 * w]
    assert (b._log.cpu().numpy()[2] == 0).all() and (b._log.cpu().numpy()[1, :, 0] == INF).all()
    assert b.total_steps() == ref.total_steps() // 4


@pytest.mark.gpu
def test_side_stream_equals_default_stream():
    import torch
    from maaco_path_planing_b200.batch import MAACOBatch
    grids = mixed_maps(64, 64, 6, 6462)
    sizes = [{"num_ants": n, "num_iterations": k} for n, k in ((256, 3), (1, 2), (31, 0), (100, 1), (33, 3), (2, 3))]
    want = MAACOBatch(grids, 8, 1, seeds=range(6), per_map_endpoints=True, map_sizes=sizes, **MAACO_DEFAULT).solve()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        got = MAACOBatch(grids, 8, 1, seeds=range(6), per_map_endpoints=True, map_sizes=sizes, **MAACO_DEFAULT).solve()
    assert got == want
    for k in range(6):
        assert want[k] == solo_solve(grids[k], sizes[k], k), k
