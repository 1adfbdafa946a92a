"""Exact Dijkstra distance fields on the GPU (mpp_dijkstra_fields / mpp_dijkstra_field_paths): fields and parents bit for
bit equal to the C oracle's whole-map Dijkstra, on single maps (a cluster of several CTAs per map) and on a batch of
300 maps (one CTA per map); paths read from them equal to the per-target searches."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from field_oracle import dijkstra_field
from test_dijkstra_field_oracle import CORNERS, field_maps, walled

pytestmark = pytest.mark.gpu

INF = float("inf")


def _batch(grids, **kw):
    from maaco_path_planing_b200.batch import SearchBatch
    return SearchBatch(np.stack(grids) if not isinstance(grids, torch.Tensor) else grids, **kw)


def _fields(sb, src=None):
    g, parent = sb._fields(src)
    return g.cpu().numpy(), parent.cpu().numpy()


def _moved(grid, rng):
    g = np.where(grid >= 2, 0, grid)
    s, t = rng.choice(np.flatnonzero(g.ravel() == 0), 2, replace=False)
    g.flat[s], g.flat[t] = 2, 3
    return g


def _assert_field(grid, src, g, parent, ad=True, rs=True, what=""):
    wg, wp = dijkstra_field(grid, src, ad, rs)
    assert np.array_equal(g.view(np.uint64), wg.view(np.uint64)), (what, int((g != wg).sum()))
    assert np.array_equal(parent, wp), (what, int((parent != wp).sum()))


@pytest.mark.parametrize("allow_diag,restrict", CORNERS)
def test_single_map_fields_equal_oracle(allow_diag, restrict):
    """One map per launch: the widest cluster per map."""
    kw = dict(allow_diagonal_moves=allow_diag, restrict_diagonal_near_obstacle_policy=restrict)
    for name, grid, src in field_maps():
        sb = _batch([grid], **kw)
        g, parent = _fields(sb, [src])
        _assert_field(grid, src, g[0], parent[0], allow_diag, restrict, name)


@pytest.mark.parametrize("shape", [(510, 510), (1022, 254), (254, 1022), (2048, 2048)])
def test_large_maps(shape):
    from maaco_path_planing_b200 import blocks_map
    grid = blocks_map(0, 0.2, seed=shape[0] + shape[1], rows=shape[0], cols=shape[1])
    srcs = [0, (shape[0] // 2) * shape[1] + shape[1] // 3]
    grid.flat[srcs[1]] = 0
    sb = _batch([grid, grid])                                 # two maps: still several CTAs per map
    g, parent = _fields(sb, srcs)
    for k, s in enumerate(srcs):
        _assert_field(grid, s, g[k], parent[k], what=(shape, s))
    assert np.isfinite(g).sum() > 0.7 * grid.size


def test_batch_of_300_maps_one_cta_each():
    """A batch of more maps than SMs (one CTA per map), each map with its own obstacles and source, some sources invalid
    (all-inf fields); a second run gives the same bits."""
    rng = np.random.default_rng(300)
    grids = [(rng.random((64, 64)) < rng.uniform(0.05, 0.35)).astype(int) for _ in range(296)]
    grids += [walled(64, 64, seed=k) for k in range(4)]
    src = np.array([int(rng.choice(np.flatnonzero(g.ravel() == 0))) for g in grids], np.int32)
    src[5], src[6] = -1, 64 * 64
    src[7] = int(np.flatnonzero(grids[7].ravel() == 1)[0])
    for ad, rs in ((True, True), (False, False)):
        sb = _batch(grids, allow_diagonal_moves=ad, restrict_diagonal_near_obstacle_policy=rs)
        g, parent = _fields(sb, torch.as_tensor(src).cuda())
        for k, grid in enumerate(grids):
            _assert_field(grid, int(src[k]), g[k], parent[k], ad, rs, k)
        assert np.isinf(g[5:8]).all()
        g2, parent2 = _fields(sb, src)
        assert np.array_equal(g.view(np.uint64), g2.view(np.uint64)) and np.array_equal(parent, parent2)


def test_distance_field_public_entry_points():
    from maaco_path_planing_b200.dijkstra import DijkstraSolver
    grid = load_golden("env_grids")["image5"].astype(int)
    s = DijkstraSolver(grid)
    f = s.distance_field()
    assert f.is_cuda and f.dtype == torch.float64 and tuple(f.shape) == grid.shape
    src = s.start_node[0] * grid.shape[1] + s.start_node[1]
    want, _ = dijkstra_field(grid, src)
    assert np.array_equal(f.cpu().numpy(), want)
    free = tuple(int(x) for x in np.argwhere(grid == 0)[100])
    want2, _ = dijkstra_field(grid, free[0] * grid.shape[1] + free[1])
    assert np.array_equal(s.distance_field(free).cpu().numpy(), want2)
    assert torch.isinf(s.distance_field((-1, 3))).all()
    sb = _batch([grid, _moved(grid, np.random.default_rng(1))])
    fs = sb.distance_fields()
    assert tuple(fs.shape) == (2,) + grid.shape
    assert np.array_equal(fs[0].cpu().numpy(), want)


def test_solve_targets_equals_a_loop_of_solve():
    from maaco_path_planing_b200.dijkstra import DijkstraSolver
    grid = walled(60, 45, seed=60)
    grid[0, 0], grid[59, 44] = 2, 3
    rng = np.random.default_rng(5)
    R, C = grid.shape
    free = [tuple(int(x) for x in p) for p in np.argwhere(grid == 0)]
    obst = [tuple(int(x) for x in p) for p in np.argwhere(grid == 1)]
    pocket = (R // 3 + 3, C // 3 + 3)                                     # inside the closed box: unreachable
    assert grid[pocket] == 0
    targets = [free[int(i)] for i in rng.integers(0, len(free), 40)] + obst[:3] + [
        (-1, 0), (R, 2), (3, C), pocket, (0, 0), None, (R - 1, C - 1)]
    for start in (None, free[77], (R, 0)):
        kw = dict(turn_penalty_factor=0.3, min_safe_distance=2.2)
        a, b = DijkstraSolver(grid, **kw), DijkstraSolver(grid, **kw)
        want = [a.solve(start, t) for t in targets]
        got = b.solve_targets(targets, start)
        assert got == want
        assert [[type(v) for v in r] for r in got] == [[type(v) for v in r] for r in want]
        assert b.convergence_curve == a.convergence_curve
        if start is None:
            assert sum(len(r[0]) > 1 for r in got) > 20 and got[-6][0] == []


def _queries(grids, per_map, rng):
    R, C = grids[0].shape
    n = len(grids) * per_map
    mi = np.repeat(np.arange(len(grids)), per_map).astype(np.int32)
    dst = rng.integers(0, R * C, n).astype(np.int32)
    starts = [int(np.flatnonzero(g.ravel() == 2)[0]) for g in grids]
    dst[::9] = [starts[m] for m in mi[::9]]
    mi[5], dst[6], dst[7] = len(grids), -1, R * C                        # outside the batch / the map: not searched
    return mi, np.array(starts, np.int32), dst


@pytest.mark.parametrize("on_device", [False, True])
def test_field_paths_equal_search(on_device):
    """128 maps of config 5's kind (256 x 256, 20 % blocks, own start and target): paths, n_cells, g and statistics
    of field_paths are the bytes of search(2, ...) from each map's start."""
    from maaco_path_planing_b200 import blocks_map
    rng = np.random.default_rng(128)
    grids = [_moved(blocks_map(256, 0.2, seed=4000 + i), rng) for i in range(128)]
    mi, starts, dst = _queries(grids, 4, rng)
    kw = dict(turn_penalty_factor=0.3, safety_penalty_factor=0.8, diagonal_obstacle_penalty_value=100.0)
    sb = _batch(torch.as_tensor(np.stack(grids)).cuda() if on_device else grids, **kw)
    want = sb.search(2, mi, starts[np.clip(mi, 0, len(grids) - 1)], dst)
    got = sb.field_paths(torch.as_tensor(mi).cuda() if on_device else mi, dst)
    w, h = [x.cpu().numpy() for x in want], [x.cpu().numpy() for x in got]
    assert np.array_equal(h[1], w[1])
    assert np.array_equal(h[2].view(np.uint64), w[2].view(np.uint64))
    assert np.array_equal(h[3].view(np.uint64), w[3].view(np.uint64))
    for i in range(len(mi)):
        assert np.array_equal(h[0][i, :h[1][i]], w[0][i, :w[1][i]]), i
    assert (h[1] > 1).sum() > len(mi) // 2 and (h[1][5:8] == 0).all()


def test_truncated_paths_grow_and_repeat():
    grids = [np.zeros((100, 100), int) for _ in range(3)]
    grids[1][40:60, 30] = 1
    for g in grids:
        g[0, 0], g[99, 99] = 2, 3
    mi = np.repeat(np.arange(3), 3).astype(np.int32)
    dst = np.array([9999, 1, 5052] * 3, np.int32)
    want = [x.cpu().numpy() for x in _batch(grids).field_paths(mi, dst)]
    sb = _batch(grids, max_cells=4)
    got = [x.cpu().numpy() for x in sb.field_paths(mi, dst)]
    assert sb.max_cells > 4 and sb.launches > 2
    for a, b in zip(got[1:], want[1:]):
        assert np.array_equal(a, b)
    for i in range(len(mi)):
        assert np.array_equal(got[0][i, :got[1][i]], want[0][i, :want[1][i]])


def test_field_follows_stream_order_on_a_side_stream():
    """The field kernel runs on torch's current stream: it sees a source written just before it on a side stream, and
    work after it on that stream sees the finished field."""
    grid = load_golden("env_grids")["image5"].astype(int)
    sb = _batch([grid])
    src = int(np.flatnonzero(grid.ravel() == 2)[0])
    want, _ = dijkstra_field(grid, src)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        s = torch.full((1,), -1, dtype=torch.int32, device="cuda")
        torch.cuda._sleep(200_000_000)                                    # keeps the side stream busy for a while
        s.fill_(src)
        f = sb.distance_fields(s)
        out = f.clone()
    side.synchronize()
    assert np.array_equal(out[0].cpu().numpy(), want)
