"""CPU checks of the whole-map Dijkstra oracle (field_oracle.py) that the GPU distance fields are compared with: at every
target T, its g and its parent chain are what the validated oracle search orc_astar(variant 2, src, T) returns."""
import numpy as np
import pytest

import pyoracle as O
from conftest import load_golden
from field_oracle import chain, dijkstra_field

CORNERS = [(True, True), (True, False), (False, True), (False, False)]   # (allow_diagonal, restrict_corner)


def walled(R, C, seed):
    """A random map with a closed box (an unreachable pocket inside it) and a wall cutting off a corner region."""
    rng = np.random.default_rng(seed)
    g = (rng.random((R, C)) < 0.15).astype(int)
    r0, c0 = R // 3, C // 3
    g[r0:r0 + 8, c0:c0 + 8] = 1
    g[r0 + 1:r0 + 7, c0 + 1:c0 + 7] = 0
    g[R - 6, C - 6:] = 1
    g[R - 6:, C - 6] = 1
    g[R - 3:, C - 3:] = 0
    return g


def field_maps():
    """(name, grid, src) of every map the field is checked on: the demo maps, image5, ragged and walled-off maps."""
    env = load_golden("env_grids")
    out = []
    for name in ("fig7", "fig13", "image1", "image2", "image3", "image5"):
        g = env[name].astype(int)
        out.append((name, g, int(np.flatnonzero(g.ravel() == 2)[0])))
    rng = np.random.default_rng(37)
    for shape in ((37, 42), (100, 150)):
        g = (rng.random(shape) < 0.25).astype(int)
        out.append((f"random{shape}", g, int(rng.choice(np.flatnonzero(g.ravel() == 0)))))
    for shape in ((20, 20), (60, 45)):
        g = walled(*shape, seed=shape[0])
        out.append((f"walled{shape}", g, 0 if g[0, 0] == 0 else int(np.flatnonzero(g.ravel() == 0)[0])))
    return out


def sampled_targets(grid, src, n, rng):
    """Every cell of a map of at most 400 cells; else n random cells, the source, obstacles and cells of other
    components."""
    size = grid.size
    if size <= 400:
        return np.arange(size)
    t = list(rng.integers(0, size, n))
    obst = np.flatnonzero(grid.ravel() == 1)
    if obst.size:
        t += list(rng.choice(obst, 8))
    return np.array(t + [src])


@pytest.mark.parametrize("allow_diag,restrict", CORNERS)
def test_field_equals_oracle_search_at_every_target(allow_diag, restrict):
    rng = np.random.default_rng(int(allow_diag) * 2 + int(restrict))
    n_unreachable = 0
    for name, grid, src in field_maps():
        g, parent = dijkstra_field(grid, src, allow_diag, restrict)
        orc = O.AStarOracle(grid, allow_diag, restrict)
        free = grid.ravel() != 1
        n_unreachable += int((free & np.isinf(g.ravel())).sum())
        assert g.flat[src] == 0.0 and parent.flat[src] == 0xFF
        assert (parent.ravel()[np.isinf(g.ravel())] == 0xFF).all()
        for T in sampled_targets(grid, src, 150, rng):
            cells, gw, _, _ = orc.solve(2, src, int(T))
            assert g.flat[T] == gw, (name, int(T), g.flat[T], gw)
            if len(cells):
                assert chain(parent, T) == cells.tolist(), (name, int(T))
            else:
                assert parent.flat[T] == 0xFF, (name, int(T))
    assert n_unreachable > 0                                  # the walled-off pockets were really unreachable


def test_invalid_source_gives_an_empty_field():
    grid = load_golden("env_grids")["fig7"].astype(int)
    obstacle = int(np.flatnonzero(grid.ravel() == 1)[0])
    for src in (obstacle, -1, grid.size):
        g, parent = dijkstra_field(grid, src)
        assert np.isinf(g).all() and (parent == 0xFF).all()
