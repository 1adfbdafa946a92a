"""SearchEngine -- the connector / fitness / statistics entry points (mpp_astar_batch_maps, mpp_waypoint_fitness_maps,
mpp_path_stats) on one map: a SearchBatch over a GridMap's one-map batch, with the reference's single-map arguments.
Populations are torch tensors in HBM; the engine only moves pointers across the C ABI.  No CPU fallback."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .batch import SearchBatch
from .gridmap import GridMap

INF = float("inf")


def make_policy(turn_penalty_factor, safety_penalty_factor, min_safe_distance, diagonal_obstacle_penalty_value,
                restrict_policy=True, allow_diagonal=True, mode=0):
    return _lib.Policy(float(turn_penalty_factor), float(safety_penalty_factor), float(min_safe_distance),
                       float(diagonal_obstacle_penalty_value), int(bool(restrict_policy)), int(bool(allow_diagonal)),
                       int(mode))


class SearchEngine(SearchBatch):
    """The searches of one map (every launch on map 0 of its batch).  Buffer sizes, their growth, the scratch and the
    longest-first order are SearchBatch's; a launch whose heap overflowed or whose paths were truncated is repeated
    whole, and `counters` adds up every launch."""

    def __init__(self, gridmap: GridMap, max_cells=None, heap_cap=None, n_slots=None, group=None):
        import torch
        super().__init__(gridmap._maps, max_cells=max_cells, heap_cap=heap_cap, n_slots=n_slots)
        self.group = group            # torch.distributed group: population batches are sharded over its ranks
        self.torch = torch
        self.map = gridmap

    def _map0(self, n):
        return self.torch.zeros(n, dtype=self.torch.int32, device=self.device)

    def _grown(self, ncell):
        return self._grow_from(*self.torch.stack([ncell.min(), ncell.max()]).tolist())

    def expansions(self):
        """(node expansions, successful relaxations) of the searches so far."""
        c = self.counters.cpu().numpy()
        return int(c[0]), int(c[1])

    def queue_stats(self):
        """(ring pushes, overflow-heap pushes) of the searches so far."""
        c = self.counters.cpu().numpy()
        return int(c[2]), int(c[3])

    # -- K5 ---------------------------------------------------------------------------------------
    def astar_batch(self, variant, src, dst, avoid_bits=None, allow_diagonal=True, restrict_corner=True):
        """n independent searches.  Returns (cells[n,max_cells], n_cells[n], g[n]) as device tensors."""
        t = self.torch
        src, dst = self._i32(src), self._i32(dst)
        n = src.numel()
        if avoid_bits is not None:
            avoid_bits = t.as_tensor(avoid_bits, device=self.device).contiguous()
            assert avoid_bits.numel() == n * self.words
        mi = self._map0(n)
        while True:
            cells, ncell, g, _ = self._launch(variant, mi, src, dst, avoid_bits, False, allow_diagonal, restrict_corner,
                                              None)
            if not self._grown(ncell):
                return cells, ncell, g

    # -- K6 + K7 ----------------------------------------------------------------------------------
    def waypoint_fitness(self, waypoints, policy):
        """waypoints: [N, W] int32 cells.  Returns (cells, n_cells, stats[N,5]) device tensors.

        With a process group, individuals are independent units: rank g evaluates rows
        [g*per, (g+1)*per) and the results are all-gathered (no other data-path collective)."""
        t = self.torch
        if self.map.start_cell < 0 or self.map.target_cell < 0:
            raise _lib.MppError("waypoint_fitness: the map has no start / target")
        wps = self._i32(waypoints)
        N, W = wps.shape
        world = 1
        if self.group is not None:
            import torch.distributed as dist
            world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if world == 1 or N < 2 * world:
            return self._waypoint_fitness_local(wps, policy)
        per = (N + world - 1) // world
        if per * world != N:                                           # pad with copies of row 0 (equal shards)
            wps = t.cat([wps, wps[:1].expand(per * world - N, W)]).contiguous()
        while True:
            cells, ncell, stats = self._waypoint_fitness_local(wps[rank * per:(rank + 1) * per].contiguous(), policy,
                                                               retry=False)
            flags = t.stack([ncell.min(), -ncell.max()]).to(t.int64)
            dist.all_reduce(flags, op=dist.ReduceOp.MIN, group=self.group)
            if self._grow_from(int(flags[0]), int(-flags[1])):
                continue                                               # every rank grows the same way and repeats
            a_cells = t.empty((per * world, cells.shape[1]), dtype=t.int32, device=self.device)
            a_ncell = t.empty(per * world, dtype=t.int32, device=self.device)
            a_stats = t.empty((per * world, 5), dtype=t.float64, device=self.device)
            dist.all_gather_into_tensor(a_cells, cells.contiguous(), group=self.group)
            dist.all_gather_into_tensor(a_ncell, ncell, group=self.group)
            dist.all_gather_into_tensor(a_stats, stats, group=self.group)
            return a_cells[:N], a_ncell[:N], a_stats[:N]

    def _waypoint_fitness_local(self, wps, policy, retry=True):
        mi = self._map0(wps.shape[0])
        while True:
            cells, ncell, stats = self._chain_launch(mi, wps, policy)
            if not retry or not self._grown(ncell):
                return cells, ncell, stats

    # -- K7 ---------------------------------------------------------------------------------------
    def path_stats(self, cells, n_cells, policy):
        """cells [P, max_cells] int32, n_cells [P] -> stats [P,5] device tensor."""
        t = self.torch
        cells = cells if isinstance(cells, t.Tensor) else t.as_tensor(np.ascontiguousarray(cells, np.int32), device=self.device)
        cells = cells.contiguous()
        ncell = self._i32(n_cells)
        P, mc = cells.shape
        stats = t.empty((P, 5), dtype=t.float64, device=self.device)
        _lib.check(_lib.lib().mpp_path_stats(self._maps, _lib.ptr(self._map0(P)), _lib.ptr(cells), mc, _lib.ptr(ncell), P,
                                             C.byref(policy), _lib.ptr(stats), self._stream()), "mpp_path_stats")
        self.launches += 1
        return stats

    def stats_of_path(self, path, policy):
        """helper.calculate_path_stats for one python path (list of (r,c)) -> 6-tuple like the reference."""
        if not path:
            return [], INF, 0, 0.0, 0.0, INF                              # helper.py:104-105
        cells = np.array([[r * self.cols + c for r, c in path]], np.int32)
        st = self.path_stats(cells, np.array([len(path)], np.int32), policy).cpu().numpy()[0]
        length = float(st[0]) if len(path) > 1 else 0
        return path, length, int(st[1]), float(st[2]), float(st[3]), float(st[4])
