"""Every sharded code path on ONE GPU: W ranks emulated by the lockstep process group (tests/lockstep_group.py), against
the single-colony oracle (or the single-GPU solvers, themselves oracle-checked) bit for bit.

The sharded MAACO colony runs kernels no single-GPU test reaches -- the tour kernel's peer-memory form, the all-gather
exchange's pack / unpack / replay kernels, the pheromone update of a slice of tile rows -- and host code that sizes the
exchange, repeats passes after an overflow and picks the exchange.  A rank's "peer" buffer is then a buffer on the same
device and an all-gather a copy, which computes exactly what W GPUs compute.  (Cross-GPU memory ordering is what this
cannot see; tests/multigpu_check.py covers it under torchrun.)

Every rank checks after every pass: all per-ant records (replicated), its own ants' tours, the whole pheromone field,
the colony's best state; and after solve_path_planning(), the path, length, turns and convergence curve.  Then it waits
at a barrier: over peer memory the next pass's tour kernels of the other ranks store into this rank's result table, so
what a rank reads of a pass is only stable until every rank has read it (with real GPUs as here)."""
import functools

import numpy as np
import pytest
import torch.distributed as dist

from conftest import MAACO_DEFAULT
from lockstep_group import lockstep_group
from test_batch_sweeps_gpu import serpentine

pytestmark = pytest.mark.gpu
INF = float("inf")
EXCHANGES = [pytest.param(True, id="peer"), pytest.param(False, id="allgather")]


def _blocks(n, seed, rows=None, cols=None):
    from maaco_path_planing_b200 import blocks_map
    return blocks_map(n, 0.2, seed=seed, rows=rows, cols=cols)


MAPS = {
    "blocks96": lambda: _blocks(96, 11),                     # 3 tile rows: from 4 ranks on, some own only padding
    "ragged100x150": lambda: _blocks(0, 0, rows=100, cols=150),
    "blocks128": lambda: _blocks(128, 12),
    "blocks64": lambda: _blocks(64, 7),
    "config4": lambda: _blocks(512, 4000),
    "serpentine48": lambda: serpentine(48),
}


@functools.lru_cache(maxsize=None)
def grid_of(name):
    return MAPS[name]()


@functools.lru_cache(maxsize=8)
def oracle_run(name, N, K, seed):
    """The oracle's colony, pass by pass: per-ant records, tours, tau and best state; then its solve."""
    import pyoracle as O
    orc = O.MaacoOracle(grid_of(name), N, K, seed=seed, threads=0, **MAACO_DEFAULT)
    passes, best_ant = [], -1
    for it in range(1, K + 1):
        before = orc.best_path
        cells, nc, ln, tn, (bi, _, _) = orc.iterate(it)
        if orc.best_path is not before:
            best_ant = int(bi)
        passes.append(dict(cells=cells[:, :max(1, int(nc.max()))].copy(), nc=nc, ln=ln, tn=tn, tau=orc.tau.copy(),
                           best=(orc.best_len, orc.best_turns, len(orc.best_path), best_ant)))
    solve = (orc.best_path.tolist(), orc.best_len, orc.best_turns if orc.best_turns >= 0 else INF, list(orc.curve))
    return passes, solve


def single_run(name, N, K, seed, **kw):
    """The same, recorded from a single-GPU MAACO (tours cut at its max_cells; solve = its result or its MppError)."""
    from maaco_path_planing_b200 import MAACO
    from maaco_path_planing_b200._lib import MppError
    dev = MAACO(grid_of(name), N, K, rng_seed=seed, device=0, verbose=False, **MAACO_DEFAULT, **kw)
    passes = []
    for it in range(1, K + 1):
        dev.run_iteration(it)
        nc, ln, tn, cells = dev.last_tours()
        st = dev._read_state()
        passes.append(dict(cells=cells, nc=nc, ln=ln, tn=tn, tau=dev.pheromone_matrix.ravel().copy(),
                           best=(st.best_len, st.best_turns, st.best_n_cells, st.best_ant)))
    try:
        path, length, turns = dev.solve_path_planning()
        solve = ([r * dev.cols + c for r, c in path], length, turns, list(dev.convergence_curve_data))
    except MppError as e:
        solve = e
    return passes, solve


def check_pass(dev, ref, tag):
    nc, ln, tn = dev.last_results()
    assert np.array_equal(nc, ref["nc"]), f"{tag}: n_cells"
    assert np.array_equal(ln, ref["ln"]), f"{tag}: lengths"
    assert np.array_equal(tn, ref["tn"]), f"{tag}: turns"
    lnc, _, _, cells = dev.last_tours()
    sl = slice(dev.ant_offset, dev.ant_offset + dev.n_local)
    assert np.array_equal(lnc, ref["nc"][sl]), f"{tag}: n_cells of the local ants"
    w = min(cells.shape[1], ref["cells"].shape[1])                   # (cells past a max_cells cut are not compared)
    mask = np.arange(w)[None, :] < lnc[:, None]
    assert np.array_equal(cells[:, :w][mask], ref["cells"][sl, :w][mask]), f"{tag}: tours of the local ants"
    assert np.array_equal(dev.pheromone_matrix.ravel(), ref["tau"]), f"{tag}: pheromone"
    st = dev._read_state()
    assert (st.best_len, st.best_turns, st.best_n_cells, st.best_ant) == ref["best"], f"{tag}: best state"


def check_solve(dev, ref, tag):
    from maaco_path_planing_b200._lib import MppError
    if isinstance(ref, MppError):
        with pytest.raises(MppError) as e:
            dev.solve_path_planning()
        assert str(e.value) == str(ref), tag
        return
    path, length, turns = dev.solve_path_planning()
    opath, olen, oturns, ocurve = ref
    assert [r * dev.cols + c for r, c in path] == list(opath), f"{tag}: path"
    assert (length, turns) == (olen, oturns), f"{tag}: length, turns"
    assert dev.convergence_curve_data == ocurve, f"{tag}: convergence curve"


def sharded(monkeypatch, W, name, N, K, seed, p2p, body, **kw):
    """body(dev, rank) on every rank of a MAACO colony sharded over W emulated ranks."""
    from maaco_path_planing_b200 import MAACO
    monkeypatch.setenv("MPP_P2P", "1" if p2p else "0")
    grid = grid_of(name)
    with lockstep_group(monkeypatch, W) as g:
        def rank(r):
            dev = MAACO(grid, N, K, rng_seed=seed, device=0, group=g, verbose=False, **MAACO_DEFAULT, **kw)
            body(dev, r)
            # (a fake that failed would silently test the other exchange; more than 16 ranks cannot use peer memory)
            assert (dev._p2p is not None) == (p2p and W <= 16), f"rank {r}: exchange ({getattr(dev, '_p2p_error', '')})"
        g.run(rank)


def passes_and_solve(ref_passes, ref_solve, W, K):
    def body(dev, r):
        for it in range(1, K + 1):
            dev.run_iteration(it)
            check_pass(dev, ref_passes[it - 1], f"rank {r}/{W} pass {it}")
            dist.barrier(group=dev.group)
        check_solve(dev, ref_solve, f"rank {r}/{W}")
    return body


# ---- against the oracle ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p2p", EXCHANGES)
@pytest.mark.parametrize("per", [13, 40, 64])         # 13, 40: ranks share words of the (tile, ant) bitmaps
@pytest.mark.parametrize("W", [2, 3, 4, 8, 16])
def test_colony_vs_oracle(monkeypatch, W, per, p2p):
    N, K, seed = per * W, 6, 9
    ref = oracle_run("blocks96", N, K, seed)
    sharded(monkeypatch, W, "blocks96", N, K, seed, p2p, passes_and_solve(*ref, W, K))


@pytest.mark.parametrize("p2p", EXCHANGES)
def test_ragged_map(monkeypatch, p2p):
    """100 x 150: a partial last tile row and tile column, 4 tile rows padded to 6 over 3 ranks."""
    W, N, K, seed = 3, 120, 5, 21
    ref = oracle_run("ragged100x150", N, K, seed)
    sharded(monkeypatch, W, "ragged100x150", N, K, seed, p2p, passes_and_solve(*ref, W, K))


@pytest.mark.parametrize("p2p", EXCHANGES)
def test_1500_ants_per_rank(monkeypatch, p2p):
    """More local ants than one 1024-thread round of the exchange's segment scan."""
    W, N, K, seed = 2, 3000, 3, 33
    ref = oracle_run("blocks128", N, K, seed)
    sharded(monkeypatch, W, "blocks128", N, K, seed, p2p, passes_and_solve(*ref, W, K))


@pytest.mark.parametrize("W", [17])
def test_more_ranks_than_peer_slots(monkeypatch, W):
    """Peer memory asked for, but the peer tour kernel takes at most 16 ranks: the all-gather exchange is used."""
    N, K, seed = 13 * W, 4, 9
    ref = oracle_run("blocks96", N, K, seed)
    sharded(monkeypatch, W, "blocks96", N, K, seed, True, passes_and_solve(*ref, W, K))


# ---- the all-gather exchange's overflow handling ----------------------------------------------------------------------
def test_exchange_capacity_zero_from_the_first_pass(monkeypatch):
    W, N, K, seed = 8, 8 * 64, 6, 9
    ref_passes, ref_solve = oracle_run("blocks96", N, K, seed)

    def body(dev, r):
        dev._cap = dev._cap_max = 0
        passes_and_solve(ref_passes, ref_solve, W, K)(dev, r)
        assert dev.exchange_rewinds >= 1, f"rank {r}: the exchange should have overflowed"
    sharded(monkeypatch, W, "blocks96", N, K, seed, False, body)


def test_rewind_after_the_capacity_changed(monkeypatch):
    """Pass 3 overflows (capacity 0) while pass 4 is already enqueued with another capacity: the repeat must size the
    exchange from pass 3's true code totals, not from a buffer pass 4 has re-gathered."""
    from maaco_path_planing_b200.maaco import _round64k
    W, per, K, seed = 8, 40, 6, 9
    N = W * per
    ref_passes, ref_solve = oracle_run("blocks96", N, K, seed)
    codes = np.maximum(ref_passes[2]["nc"].astype(np.int64) - 1, 0)
    true_max_total = int(codes.reshape(W, per).sum(axis=1).max())

    def body(dev, r):
        dev.run_iteration(1)
        dev.run_iteration(2)
        restored = dev._cap_max
        dev._cap_max = 0
        dev.run_iteration(3)                                         # sized when pass 1 is confirmed: capacity 0
        dev._cap_max = restored
        dev.run_iteration(4)                                         # sized from pass 2: a non-zero capacity
        check_pass(dev, ref_passes[3], f"rank {r}/{W} pass 4")
        dist.barrier(group=dev.group)
        assert dev.exchange_rewinds == 1, f"rank {r}"
        assert dev._cap_max == max(restored, _round64k(2 * true_max_total)), f"rank {r}: capacity after the rewind"
        for it in range(5, K + 1):
            dev.run_iteration(it)
            check_pass(dev, ref_passes[it - 1], f"rank {r}/{W} pass {it}")
            dist.barrier(group=dev.group)
        check_solve(dev, ref_solve, f"rank {r}/{W}")
    sharded(monkeypatch, W, "blocks96", N, K, seed, False, body)


@pytest.mark.parametrize("p2p", EXCHANGES)
@pytest.mark.parametrize("name, max_cells", [("serpentine48", None), ("blocks64", 16)], ids=["serpentine", "explicit16"])
def test_tours_longer_than_max_cells(monkeypatch, p2p, name, max_cells):
    """Tours that do not fit max_cells: per-ant records and tau stay exact (the all-gather exchange grows its move
    buffers and repeats the pass), and the solve behaves as on one GPU -- the serpentine's 1175-cell path through a
    repeat at full capacity, an explicit max_cells as the same MppError."""
    W, N, K, seed = 2, 32, 3, 5
    kw = {} if max_cells is None else dict(max_cells=max_cells)
    ref = single_run(name, N, K, seed, **kw)
    if max_cells is None:
        assert len(ref[1][0]) == 1175                                # the best path is longer than the default
    sharded(monkeypatch, W, name, N, K, seed, p2p, passes_and_solve(*ref, W, K), **kw)


# ---- against the single-GPU colony (oracle-checked at this size by test_maaco_gpu.py) ----------------------------------
@pytest.mark.parametrize("p2p", EXCHANGES)
def test_config4_vs_single_gpu(monkeypatch, p2p):
    """BASELINE config 4: 4096 ants on 512 x 512 (16 tile rows, 2 per rank), 2 passes."""
    W, N, K, seed = 8, 4096, 2, 4
    ref = single_run("config4", N, K, seed)
    sharded(monkeypatch, W, "config4", N, K, seed, p2p, passes_and_solve(*ref, W, K))


# ---- sharded populations of PSO, GA and MPA (what tests/multigpu_solvers_check.py runs under torchrun) -----------------
POLICY = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, min_safe_distance=1.8,
              diagonal_obstacle_penalty_value=100.0, allow_diagonal_moves=True,
              restrict_diagonal_near_obstacle_policy=True)


@pytest.mark.parametrize("W", [3, 8])
def test_sharded_populations_vs_goldens(monkeypatch, W):
    """33 particles / chromosomes (padded shards) and 20 predators over 8 ranks (one rank owns none)."""
    import os
    from conftest import GOLDEN
    from maaco_path_planing_b200.ga_solver import GASolver
    from maaco_path_planing_b200.mpa import MPA
    from maaco_path_planing_b200.pso import PSOSolver
    gold = np.load(os.path.join(GOLDEN, "solver_cases.npz"))

    with lockstep_group(monkeypatch, W) as grp:
        def rank(r):
            for name in ("fig7_33", "blocks40_33"):
                k = "pso_" + name
                N, K, seed = (int(x) for x in gold[k + "_meta"])
                grid = gold[k + "_grid"].astype(int)
                s = PSOSolver(grid, num_iterations=K, num_particles=N, num_waypoints_per_particle=5, w=0.7, c1=1.5,
                              c2=1.5, rng_seed=seed, device=0, verbose=False, group=grp, **POLICY)
                res = s.solve()
                assert np.array_equal(np.array(s.convergence_curve), gold[k + "_curve"]), f"rank {r} {k}: curve"
                assert np.array_equal(s._state["pos"].cpu().numpy(), gold[k + "_pos"]), f"rank {r} {k}: positions"
                C = grid.shape[1]
                assert np.array_equal(np.array([a * C + b for a, b in res[0]], np.int32), gold[k + "_best"]), k
                k = "ga_" + name
                N, K, seed = (int(x) for x in gold[k + "_meta"])
                ga = GASolver(grid, num_generations=K, population_size=N, num_waypoints_per_chromosome=5,
                              mutation_rate=0.1, crossover_rate=0.8, tournament_size=3, rng_seed=seed, device=0,
                              verbose=False, group=grp, **POLICY)
                ga.solve()
                assert np.array_equal(np.array(ga.convergence_curve), gold[k + "_curve"]), f"rank {r} {k}: curve"
                assert np.array_equal(ga._pop["chrom"].cpu().numpy(), gold[k + "_chrom"]), f"rank {r} {k}: population"
            for name in ("fig7_20", "blocks40_24"):
                k = "mpa_" + name
                N, K, seed, beta10 = (int(x) for x in gold[k + "_meta"])
                grid = gold[k + "_grid"].astype(int)
                m = MPA(grid, num_predators=N, num_iterations=K, FADs_rate=0.2, P_const=0.5, levy_beta=beta10 / 10.0,
                        turn_penalty_factor=0.1, safety_penalty_factor=0.8, min_safe_distance=1.8,
                        diagonal_obstacle_penalty=100.0, rng_seed=seed, device=0, verbose=False, group=grp)
                m.solve_path_planning()
                curve = np.array([np.inf if v is None else v for v in m.convergence_curve_data])
                assert np.array_equal(curve, gold[k + "_curve"]), f"rank {r} {k}: curve"
                assert np.array_equal(m._pop["stats"][:, 4].cpu().numpy(), gold[k + "_pop_fit"]), f"rank {r} {k}: population"
        grp.run(rank)
