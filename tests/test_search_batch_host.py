"""Host-side checks of the batched A* / Dijkstra over maps (no GPU needed): the reference's errors for maps without a
start or target, grouping of maps into waves by shape, validation of queries."""
import numpy as np
import pytest
import torch

from maaco_path_planing_b200.batch import _check_endpoints, _shape_waves, _valid_queries, solve_search_batch


def _grid(rows=6, cols=7, start=True, target=True):
    g = np.zeros((rows, cols), int)
    if start:
        g[0, 0] = 2
    if target:
        g[rows - 1, cols - 1] = 3
    return g


@pytest.mark.parametrize("algorithm,start_msg,target_msg", [
    ("astar", "AStar: Start node not found in grid.", "AStar: Target node not found in grid."),
    ("dijkstra", "Dijkstra: Start node not found.", "Dijkstra: Target node not found."),
])
def test_missing_start_or_target_raises_reference_error(algorithm, start_msg, target_msg):
    # raised before any device work: this runs without a GPU
    for grids, msg in (([_grid(), _grid(start=False)], start_msg),
                       ([_grid(), _grid(target=False)], target_msg),
                       ([_grid(start=False, target=False)], start_msg),            # start is checked first (astar.py:19)
                       ([_grid(target=False), _grid(start=False)], target_msg)):  # the first bad map decides
        with pytest.raises(ValueError) as e:
            solve_search_batch(grids, algorithm, {})
        assert str(e.value) == msg
        with pytest.raises(ValueError) as e:
            _check_endpoints(np.stack(grids).reshape(len(grids), -1), algorithm)
        assert str(e.value) == msg
    _check_endpoints(np.stack([_grid(), _grid()]).reshape(2, -1), algorithm)


def test_unknown_algorithm_is_rejected():
    with pytest.raises(ValueError, match="astar"):
        solve_search_batch([_grid()], "bfs", {})


def test_waves_group_maps_by_shape():
    grids = [_grid(6, 7), _grid(5, 5), _grid(6, 7), _grid(6, 7), _grid(5, 5), _grid(9, 4), _grid(6, 7)]
    assert _shape_waves(grids, 0, len(grids)) == [[0, 2, 3, 6], [1, 4], [5]]           # default: one wave per shape
    assert _shape_waves(grids, 0, len(grids), 3) == [[0, 2, 3], [6], [1, 4], [5]]
    assert _shape_waves(grids, 0, len(grids), 1) == [[i] for i in (0, 2, 3, 6, 1, 4, 5)]
    assert _shape_waves(grids, 2, 5) == [[2, 3], [4]]                                 # a rank's shard [lo, hi)
    assert _shape_waves(grids, 3, 3) == []


def test_query_validation():
    t = torch.tensor
    ok = _valid_queries(t([0, 1, 2, -1, 3, 0, 0, 0, 0]), t([0, 5, 41, 0, 0, -1, 42, 0, 7]),
                        t([41, 5, 0, 0, 0, 0, 0, 42, -3]), n_maps=3, n_cells=42)
    assert ok.tolist() == [True, True, True, False, False, False, False, False, False]
    with pytest.raises(ValueError, match="length"):
        _valid_queries(t([0, 1]), t([0, 1, 2]), t([0, 1]), 3, 42)
    with pytest.raises(ValueError, match="length"):
        _valid_queries(t([0, 1]), t([0, 1]), t([0]), 3, 42)
    with pytest.raises(ValueError, match="1-D"):
        _valid_queries(t([[0, 1]]), t([[0, 1]]), t([[0, 1]]), 3, 42)
