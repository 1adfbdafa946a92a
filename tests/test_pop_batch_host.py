"""Host-side checks of PSO / GA over batches of maps (no GPU needed): the reference's errors for maps without a start or
target, grouping of maps into waves by shape and rank shard, validation of seeds and grids -- all before device work."""
import numpy as np
import pytest

from maaco_path_planing_b200.batch import (GABatch, PSOBatch, _pop_waves, default_pop_wave, solve_ga_batch,
                                           solve_pso_batch)


def _grid(rows=6, cols=7, start=True, target=True):
    g = np.zeros((rows, cols), int)
    if start:
        g[0, 0] = 2
    if target:
        g[rows - 1, cols - 1] = 3
    return g


PSO_ARGS = (3, 8, 2, 0.7, 1.5, 1.5)              # iterations, particles, waypoints, w, c1, c2
GA_ARGS = (3, 8, 2, 0.1, 0.8)                    # generations, population, waypoints, mutation, crossover


def _sweep(planner, grids, **kw):
    if planner == "pso":
        return solve_pso_batch(grids, 3, 8, 2, dict(w=0.7, c1=1.5, c2=1.5), **kw)
    return solve_ga_batch(grids, 3, 8, 2, dict(mutation_rate=0.1, crossover_rate=0.8), **kw)


@pytest.mark.parametrize("planner,cls,args,name", [("pso", PSOBatch, PSO_ARGS, "PSO"), ("ga", GABatch, GA_ARGS, "GA")])
def test_missing_start_or_target_raises_reference_error(planner, cls, args, name):
    start_msg, target_msg = f"{name}: Start node not found.", f"{name}: Target node not found."   # pso.py / ga_solver.py:19-20
    for grids, msg in (([_grid(), _grid(start=False)], start_msg),
                       ([_grid(), _grid(target=False)], target_msg),
                       ([_grid(start=False, target=False)], start_msg),
                       ([_grid(target=False), _grid(start=False)], target_msg)):      # the first bad map decides
        with pytest.raises(ValueError) as e:
            cls(np.stack(grids), *args)
        assert str(e.value) == msg
        with pytest.raises(ValueError) as e:
            _sweep(planner, grids)
        assert str(e.value) == msg


@pytest.mark.parametrize("cls,args", [(PSOBatch, PSO_ARGS), (GABatch, GA_ARGS)])
def test_seeds_and_grids_are_validated(cls, args):
    grids = np.stack([_grid(), _grid(), _grid()])
    with pytest.raises(ValueError, match="seeds"):
        cls(grids, *args, seeds=[1, 2])
    with pytest.raises(ValueError, match="n_maps, rows, cols"):
        cls(_grid(), *args)
    with pytest.raises(ValueError, match="n_maps, rows, cols"):
        cls(grids[None], *args)


def test_waves_group_maps_by_shape_and_shard(monkeypatch):
    import torch.distributed as dist
    from maaco_path_planing_b200.batch import shard_maps
    grids = [_grid(6, 7), _grid(5, 5), _grid(6, 7), _grid(6, 7), _grid(5, 5), _grid(9, 4), _grid(6, 7)]
    assert _pop_waves(grids, 0, len(grids), 8, 3) == [[0, 2, 3], [6], [1, 4], [5]]
    assert _pop_waves(grids, 0, len(grids), 8) == [[0, 2, 3, 6], [1, 4], [5]]          # default: all of a small shape
    monkeypatch.setattr(dist, "get_world_size", lambda group: 2)
    shards = []
    for rank in (0, 1):
        monkeypatch.setattr(dist, "get_rank", lambda group, r=rank: r)
        lo, hi = shard_maps(len(grids), group=object())
        shards.append(_pop_waves(grids, lo, hi, 8, 2))
    assert shards == [[[0, 2], [3], [1]], [[4], [5], [6]]]                             # ranks own maps 0-3 and 4-6


def test_default_wave_bounds_the_population_paths():
    assert default_pop_wave(256, 256, 1024) == 32                       # 32 maps x 1024 x 8192 cells x 4 B = 1 GiB
    assert default_pop_wave(256, 256, 4096) == 8
    assert default_pop_wave(1000, 1000, 10 ** 6) == 1
    for shape, pop in (((64, 64), 256), ((100, 100), 1024), ((512, 512), 4096)):
        n = shape[0] * shape[1]
        mc = min(n, max(4096, 16 * sum(shape)))
        assert default_pop_wave(*shape, pop) * pop * mc * 4 <= 1 << 30
