"""The connector, waypoint-fitness and MPA kernels on both sides of their shared-memory staging limits (occupancy staged
without the opt-in attribute, staged with it, read through L2), and the batched solvers on tall and wide maps, against
the oracle bit for bit.  The shapes and their checks are in tests/smem_tiers_check.py, which also runs the 32 KB maps
in a process of their own."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import MAACO_DEFAULT, ROOT
from smem_tiers_check import AT_LIMIT, SHAPES, check_connectors, check_fitness, check_mpa, check_mpa_batch, \
    check_occ_bytes, check_pso_ga, grid_of

pytestmark = pytest.mark.gpu

SHAPE_IDS = [f"{r}x{c}" for r, c, _, _ in SHAPES]
RECT = [s for s in AT_LIMIT if s[0] != s[1]]


@pytest.mark.parametrize("rows,cols,nbytes,tier", SHAPES, ids=SHAPE_IDS)
def test_shape_has_its_occupancy_bytes(rows, cols, nbytes, tier):
    check_occ_bytes(rows, cols, nbytes)


@pytest.mark.parametrize("rows,cols,nbytes,tier", SHAPES, ids=SHAPE_IDS)
def test_connectors_vs_oracle(rows, cols, nbytes, tier):
    check_connectors(grid_of(rows, cols))


@pytest.mark.parametrize("rows,cols,nbytes,tier", SHAPES, ids=SHAPE_IDS)
def test_waypoint_fitness_vs_oracle(rows, cols, nbytes, tier):
    check_fitness(grid_of(rows, cols), stats_modes=(rows, cols) == (510, 510))


@pytest.mark.parametrize("rows,cols,nbytes,tier", SHAPES, ids=SHAPE_IDS)
def test_mpa_solo_vs_oracle_and_batch_vs_solo(rows, cols, nbytes, tier):
    check_mpa_batch(rows, cols, first=check_mpa(grid_of(rows, cols)))


def test_pso_ga_on_a_32kb_map_vs_oracle():
    check_pso_ga(grid_of(510, 510))


def test_32kb_maps_first_in_a_fresh_process():
    """No earlier launch in this process can have raised a kernel's shared-memory limit for the 32 KB maps."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "smem_tiers_check.py")], capture_output=True,
                         text=True, timeout=900)
    assert out.returncode == 0 and "smem_tiers_check ok" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]


@pytest.mark.parametrize("rows,cols", RECT, ids=[f"{r}x{c}" for r, c in RECT])
def test_maaco_batch_on_tall_and_wide_maps_vs_oracle(rows, cols):
    """Every pass's per-ant records and pheromone field of each map == the oracle's."""
    import pyoracle as O
    from maaco_path_planing_b200.batch import MAACOBatch
    grids = [grid_of(rows, cols, k) for k in range(2)]
    N, K, seeds = 128, 2, [3, 4]
    b = MAACOBatch(np.stack(grids), N, K, seeds=seeds, **MAACO_DEFAULT)
    assert (b.rows, b.cols) == (rows, cols)
    orcs = [O.MaacoOracle(g, N, K, seed=s, threads=0, **MAACO_DEFAULT) for g, s in zip(grids, seeds)]
    for it in range(1, K + 1):
        b.run_iteration(it)
        nc, ln, tn = b.last_results()
        tau = b.pheromone()
        for k, orc in enumerate(orcs):
            _, onc, oln, otn, _ = orc.iterate(it)
            assert np.array_equal(nc[k], onc) and np.array_equal(ln[k], oln) and np.array_equal(tn[k], otn), (k, it)
            assert np.array_equal(tau[k].ravel(), orc.tau), (k, it)
        assert (nc > 0).sum() > N // 2                                   # many tours reach the target


@pytest.mark.parametrize("planner", ["pso", "ga"])
@pytest.mark.parametrize("rows,cols", RECT, ids=[f"{r}x{c}" for r, c in RECT])
def test_pso_ga_batch_on_tall_and_wide_maps_equal_per_map_solvers(planner, rows, cols):
    """3 maps, each with its own start and target."""
    from test_pop_batch_gpu import _batch, _check_rows, _moved
    rng = np.random.default_rng(rows)
    grids = [_moved(grid_of(rows, cols, k), rng) for k in range(3)]
    K, N, W, seeds = 2, 32, 3, [51, 52, 53]
    b = _batch(planner, grids, K, N, W, seeds)
    res = b.solve()
    _check_rows(planner, b, res, grids, K, N, W, seeds)
    assert all(len(r[0]) > 0 for r in res)
