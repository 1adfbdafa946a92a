"""DijkstraSolver -- drop-in for dijkstra.DijkstraSolver (dijkstra.py:10-97): the connector kernel with a
zero heuristic (variant 2), i.e. extract-min over (g, r, c).  `distance_field` and `solve_targets` are the B200
additions: one exact distance field from a start serves any number of targets (field.py)."""
from __future__ import annotations

import numpy as np

from .astar import AStarSolver
from .field import dijkstra_fields, field_paths
from .gridmap import START_NODE_VAL, TARGET_NODE_VAL
from .helper import INF, BasePathfinder


class DijkstraSolver(AStarSolver):
    _variant = 2

    def __init__(self, grid, turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5,
                 allow_diagonal_moves=True, restrict_diagonal_near_obstacle_policy=True,
                 diagonal_obstacle_penalty_value=1000.0, *, device=None, gridmap=None, engine=None):
        g = np.asarray(grid)
        s = np.argwhere(g == START_NODE_VAL)
        t = np.argwhere(g == TARGET_NODE_VAL)
        if not s.size > 0:
            raise ValueError("Dijkstra: Start node not found.")                # dijkstra.py:19
        if not t.size > 0:
            raise ValueError("Dijkstra: Target node not found.")               # dijkstra.py:20
        BasePathfinder.__init__(self, grid, tuple(s[0]), tuple(t[0]), turn_penalty_factor, safety_penalty_factor,
                                min_safe_distance, allow_diagonal_moves, restrict_diagonal_near_obstacle_policy,
                                diagonal_obstacle_penalty_value, device=device, gridmap=gridmap, engine=engine)
        self.astar_strictly_restricts_corners = self.restrict_diagonal_near_obstacle_policy
        self.dijkstra_strictly_restricts_corners = self.restrict_diagonal_near_obstacle_policy

    def _inb(self, n):
        return 0 <= n[0] < self.rows and 0 <= n[1] < self.cols

    def _field(self, start_node):
        """(the map's one-map batch, g, parent) of the field from start_node (None: the grid's start)."""
        s = start_node if start_node else self.start_node                     # (as solve() reads its override)
        src = self._cell(s) if self._inb(s) else -1                           # -1: an all-inf field
        batch = self.map.handle
        g, parent = dijkstra_fields(self.engine, batch, (1, self.rows, self.cols), self.engine._i32([src]),
                                    self.allow_diagonal_moves, self.dijkstra_strictly_restricts_corners)
        return batch, g, parent

    def distance_field(self, start_node=None):
        """[rows, cols] float64 CUDA tensor: for every cell, the g that solve(start_node, cell) appends to
        convergence_curve when it finds a path (0 at the start, +inf at obstacles and unreachable cells; all +inf when
        the start is outside the map or an obstacle)."""
        return self._field(start_node)[1][0]

    def solve_targets(self, targets, start_node=None):
        """[solve(start_node, t) for t in targets] -- the same results, appended to convergence_curve the same way --
        from one distance field and one path-reading launch."""
        s = start_node if start_node else self.start_node
        targets = [t if t else self.target_node for t in targets]             # (solve's override rule)
        q = [i for i, t in enumerate(targets) if self._inb(s) and self._inb(t)]   # the others get [] (as in solve)
        res = {}
        if q:
            batch, g, parent = self._field(s)
            mi = self.engine._i32(np.zeros(len(q)))
            dst = self.engine._i32([self._cell(targets[i]) for i in q])
            cells, ncell, gout, stats = field_paths(self.engine, batch, g, parent, mi, dst, self.policy)
            cells, ncell, gout, stats = cells.cpu().numpy(), ncell.cpu().numpy(), gout.cpu().numpy(), stats.cpu().numpy()
            res = {i: (cells[j, :ncell[j]], float(gout[j]), stats[j]) for j, i in enumerate(q)}
        out = []
        for i in range(len(targets)):
            if i not in res or len(res[i][0]) == 0:
                out.append(([], INF, 0, 0.0, 0.0, INF))                        # helper.py:104-105
                continue
            path, gi, st = self._nodes(res[i][0]), res[i][1], res[i][2]
            if len(path) > 1:
                self.convergence_curve.append(gi)                              # (as solve appends it)
            out.append((path, float(st[0]) if len(path) > 1 else 0, int(st[1]), float(st[2]), float(st[3]),
                        float(st[4])))
        return out
