"""MPA -- drop-in for MPA.MPA (MPA.py:9-464).  The predator population (variable-length paths) lives
in HBM; each iteration's phase move + memory + FADs step is one kernel launch (mpp_mpa_iteration_batch on the map
as a batch of one), the stable sorts and the best-so-far cascade (MPA.py:412-437) stay on the host."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _lib
from .engine import SearchEngine, make_policy
from .gridmap import GridMap, START_NODE_VAL, TARGET_NODE_VAL
from .maaco import _fresh_seed

INF = float("inf")


class MPA:
    def __init__(self, grid, num_predators, num_iterations, FADs_rate=0.2, P_const=0.5, levy_beta=1.5,
                 turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5,
                 allow_diagonal_moves=True, restrict_diagonal_near_obstacle=True, diagonal_obstacle_penalty=1000.0,
                 *, rng_seed=None, device=None, verbose=True, group=None):
        self.grid = np.array(grid, dtype=int)                           # MPA.py:20
        self.rows, self.cols = self.grid.shape
        self.num_predators = num_predators
        self.num_iterations = num_iterations
        self.FADs_rate, self.P_const, self.levy_beta = FADs_rate, P_const, levy_beta
        self.turn_penalty_factor_mpa = turn_penalty_factor
        self.safety_penalty_factor_mpa = safety_penalty_factor
        self.min_safe_distance_mpa = min_safe_distance
        self.allow_diagonal_moves = allow_diagonal_moves
        self.restrict_diagonal_near_obstacle = restrict_diagonal_near_obstacle
        self.diagonal_obstacle_penalty_val = diagonal_obstacle_penalty
        s = np.argwhere(self.grid == START_NODE_VAL)
        t = np.argwhere(self.grid == TARGET_NODE_VAL)
        if not s.size > 0:
            raise ValueError("MPA: Start node not found in grid.")      # MPA.py:36-37
        if not t.size > 0:
            raise ValueError("MPA: Target node not found in grid.")     # MPA.py:38-39
        self.start_node = (int(s[0][0]), int(s[0][1]))
        self.target_node = (int(t[0][0]), int(t[0][1]))
        self.obstacle_nodes = np.argwhere(self.grid == 1)
        self.best_path_overall = []
        self.best_path_length_overall = INF
        self.best_path_turns_overall = INF
        self.best_safety_penalty_overall = INF
        self.best_diag_penalty_overall = INF
        self.best_fitness_overall = INF
        self.convergence_curve_data = []
        self.rng_seed = _fresh_seed() if rng_seed is None else int(rng_seed)
        self.verbose = verbose
        self.group = group          # predators are independent given the sorted old population: sharded over ranks
        self.map = GridMap(self.grid, device=device)
        self.engine = SearchEngine(self.map)
        self._seeds = self.engine.torch.from_numpy(np.array([self.rng_seed & (2 ** 64 - 1)], np.uint64).view(np.int64)
                                                   ).to(self.engine.device)
        self._queue = self.engine.torch.zeros(1, dtype=self.engine.torch.int32, device=self.engine.device)
        self.policy = make_policy(turn_penalty_factor, safety_penalty_factor, min_safe_distance,
                                  diagonal_obstacle_penalty, restrict_diagonal_near_obstacle, allow_diagonal_moves, mode=1)
        # Levy sigma MPA.py:251-253 (constant per solver; evaluated with the reference's own expression)
        b = levy_beta
        num = math.gamma(1 + b) * math.sin(math.pi * b / 2)
        den = math.gamma((1 + b) / 2) * b * (2 ** ((b - 1) / 2))
        sig = (num / den) ** (1 / b) if den > 1e-9 else 1.0
        if isinstance(sig, complex):
            raise ValueError("levy_beta gives a complex Levy sigma in the reference expression (MPA.py:253)")
        self._levy_sigma = float(sig)
        self.predator_evaluations = 0
        self._pop = None
        self._initialize_population_with_safety()

    def _cell(self, n):
        return int(n[0]) * self.cols + int(n[1])

    def _nodes(self, cells):
        return [(int(c) // self.cols, int(c) % self.cols) for c in cells]

    def _a_star(self, start_node, end_node, nodes_to_avoid_in_path=None):   # MPA.py:106-151 (single query)
        bits = None
        if nodes_to_avoid_in_path:
            b = np.zeros(self.engine.words, np.uint32)
            for r, c in nodes_to_avoid_in_path:
                j = int(r) * self.cols + int(c)
                b[j >> 5] |= np.uint32(1 << (j & 31))
            bits = b.view(np.int32)[None, :]
        inb = lambda n: 0 <= n[0] < self.rows and 0 <= n[1] < self.cols
        if start_node == end_node:
            return [start_node], 0
        if not inb(start_node) or not inb(end_node):
            return [], INF
        cells, ncell, g = self.engine.astar_batch(1, [self._cell(start_node)], [self._cell(end_node)], bits,
                                                  self.allow_diagonal_moves, self.restrict_diagonal_near_obstacle)
        n = int(ncell[0])
        return (self._nodes(cells[0, :n].cpu().numpy()), float(g[0])) if n > 0 else ([], INF)

    def _calculate_path_stats(self, path):                                  # MPA.py:215-229
        return self.engine.stats_of_path(list(path), self.policy)

    def _initialize_population_with_safety(self):                           # MPA.py:231-245: N identical S->T searches
        t = self.engine.torch
        path, _ = self._a_star(self.start_node, self.target_node)
        if not path:
            tr, tc = self.target_node
            path = [self.start_node, self.target_node] if self.grid[tr, tc] != 1 else [self.start_node]   # :236
        st = self._calculate_path_stats(path)
        N = self.num_predators
        mc = self.engine.max_cells
        cells = t.zeros((N, mc), dtype=t.int32, device=self.engine.device)
        row = t.as_tensor(np.array([self._cell(p) for p in path], np.int32), device=self.engine.device)
        cells[:, :len(path)] = row
        ncell = t.full((N,), len(path), dtype=t.int32, device=self.engine.device)
        stats = t.as_tensor(np.array([[float(st[1]), float(st[2]), float(st[3]), float(st[4]), float(st[5])]] * N),
                            device=self.engine.device)
        self._pop = dict(cells=cells, ncell=ncell, stats=stats)

    def _individual(self, i):
        P = self._pop
        st = P["stats"][i].cpu().numpy()
        n = int(P["ncell"][i])
        return {'path': self._nodes(P["cells"][i, :n].cpu().numpy()), 'length': float(st[0]) if n > 1 else 0,
                'turns': int(st[1]), 'safety_penalty': float(st[2]), 'diag_penalty': float(st[3]), 'fitness': float(st[4])}

    @property
    def population(self):
        return [self._individual(i) for i in range(self.num_predators)]

    def _sort(self):
        t = self.engine.torch
        P = self._pop
        order = t.sort(P["stats"][:, 4], stable=True).indices
        self._pop = dict(cells=P["cells"][order].contiguous(), ncell=P["ncell"][order].contiguous(),
                         stats=P["stats"][order].contiguous())

    def _iteration(self, it, phase, CF):
        t = self.engine.torch
        eng = self.engine
        N = self.num_predators
        world, rank = 1, 0
        if self.group is not None:
            import torch.distributed as dist
            world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        per = (N + world - 1) // world
        lo, hi = min(N, rank * per), min(N, (rank + 1) * per)
        while True:
            P = self._pop
            mc = P["cells"].shape[1]
            scratch, slots = eng._scratch_for(max(1, hi - lo))
            out_cells = t.empty((per * world, mc), dtype=t.int32, device=eng.device)
            out_n = t.empty(per * world, dtype=t.int32, device=eng.device)
            out_stats = t.empty((per * world, 5), dtype=t.float64, device=eng.device)
            tmp = t.empty((slots, mc), dtype=t.int32, device=eng.device)
            avoid = t.empty((slots, eng.words), dtype=t.int32, device=eng.device)
            status = t.zeros(1, dtype=t.int32, device=eng.device)
            _lib.check(_lib.lib().mpp_mpa_iteration_batch(
                self.map.handle, C.byref(self.policy), N, lo, hi, it, phase, self.P_const, CF, self.FADs_rate,
                self._levy_sigma, self.levy_beta, _lib.ptr(self._seeds), None, _lib.ptr(P["cells"]), _lib.ptr(P["ncell"]),
                _lib.ptr(P["stats"]), mc, _lib.ptr(out_cells), _lib.ptr(out_n), _lib.ptr(out_stats), _lib.ptr(tmp),
                _lib.ptr(avoid), _lib.ptr(scratch), scratch.numel(), slots, eng.heap_cap, _lib.ptr(self._queue),
                _lib.ptr(status), _lib.ptr(eng.counters), eng._stream()), "mpp_mpa_iteration_batch")
            eng.launches += 1
            if world > 1:
                dist.all_reduce(status, op=dist.ReduceOp.MAX, group=self.group)
            st = int(status.item())
            if st == 0:
                if world > 1:                                          # in-place all-gather of the ranks' row blocks
                    sl = slice(rank * per, (rank + 1) * per)
                    dist.all_gather_into_tensor(out_cells, out_cells[sl], group=self.group)
                    dist.all_gather_into_tensor(out_n, out_n[sl], group=self.group)
                    dist.all_gather_into_tensor(out_stats, out_stats[sl], group=self.group)
                self._pop = dict(cells=out_cells[:N], ncell=out_n[:N], stats=out_stats[:N])
                self.predator_evaluations += N
                return
            if st == 1:
                if eng.heap_cap >= 8 * eng.n:
                    raise _lib.MppError("A* heap overflow at maximum capacity")
                eng.heap_cap = min(8 * eng.n, eng.heap_cap * 4)
            else:
                new_mc = min(2 * eng.n, 2 * mc)
                if new_mc == mc:
                    raise _lib.MppError("path buffer overflow at maximum capacity")
                self._pop["cells"] = t.nn.functional.pad(P["cells"], (0, new_mc - mc))
                eng.max_cells = new_mc

    def solve_path_planning(self):                                          # MPA.py:320-448
        K = self.num_iterations
        self._sort()
        e = self._individual(0)
        self.best_path_overall = list(e['path'])
        self.best_path_length_overall = e['length']
        self.best_path_turns_overall = e['turns']
        self.best_safety_penalty_overall = e['safety_penalty']
        self.best_diag_penalty_overall = e['diag_penalty']
        self.best_fitness_overall = e['fitness']
        self.convergence_curve_data.append(self.best_fitness_overall if self.best_fitness_overall != INF else None)
        for it in range(1, K + 1):
            self._sort()                                                    # :333
            ratio = it / K
            CF = 0.0 if ratio >= 1.0 else ((1.0 - ratio) ** (2.0 * ratio) if ratio > 0 else 1.0)   # :336
            phase = 1 if it <= K / 3 else (2 if it <= 2 * K / 3 else 3)
            self._iteration(it, phase, CF)
            self._sort()                                                    # :412
            cur = self._individual(0)
            if cur['fitness'] < self.best_fitness_overall:                  # :415-421
                self._update_best_overall(cur)
            elif abs(cur['fitness'] - self.best_fitness_overall) < 1e-9:    # :422-437 tie-breaking cascade
                eq = lambda a, b: abs(a - b) < 1e-9
                if cur['length'] < self.best_path_length_overall:
                    self._update_best_overall(cur)
                elif eq(cur['length'], self.best_path_length_overall) and cur['turns'] < self.best_path_turns_overall:
                    self._update_best_overall(cur)
                elif eq(cur['length'], self.best_path_length_overall) and eq(cur['turns'], self.best_path_turns_overall) \
                        and cur['safety_penalty'] < self.best_safety_penalty_overall:
                    self._update_best_overall(cur)
                elif eq(cur['length'], self.best_path_length_overall) and eq(cur['turns'], self.best_path_turns_overall) \
                        and eq(cur['safety_penalty'], self.best_safety_penalty_overall) \
                        and cur['diag_penalty'] < self.best_diag_penalty_overall:
                    self._update_best_overall(cur)
            self.convergence_curve_data.append(
                self.best_fitness_overall if self.best_fitness_overall != INF else
                (self.convergence_curve_data[-1] if self.convergence_curve_data and self.convergence_curve_data[-1] is not None else None))
            if self.verbose and (it % 10 == 0 or it == 1 or it == K):
                print(f"MPA Iter {it}/{K}: IterBest L={cur['length']:.2f},T={cur['turns']},SP={cur['safety_penalty']:.2f},"
                      f"DP={cur['diag_penalty']:.2f},Fit={cur['fitness']:.2f}; OverallBest L={self.best_path_length_overall:.2f},"
                      f"T={self.best_path_turns_overall},SP={self.best_safety_penalty_overall:.2f},"
                      f"DP={self.best_diag_penalty_overall:.2f},Fit={self.best_fitness_overall:.2f}")
        if self.verbose:
            if self.best_path_overall:
                print(f"\nMPA Solved: Fitness={self.best_fitness_overall:.2f} (L={self.best_path_length_overall:.2f},"
                      f"T={self.best_path_turns_overall},SP={self.best_safety_penalty_overall:.2f},DP={self.best_diag_penalty_overall:.2f})")
            else:
                print("\nMPA: No solution found.")
        return (self.best_path_overall, self.best_path_length_overall, self.best_path_turns_overall,
                self.best_safety_penalty_overall, self.best_diag_penalty_overall, self.best_fitness_overall)

    def _update_best_overall(self, new_best_obj):                           # MPA.py:450-457
        self.best_fitness_overall = new_best_obj['fitness']
        self.best_path_overall = list(new_best_obj['path'])
        self.best_path_length_overall = new_best_obj['length']
        self.best_path_turns_overall = new_best_obj['turns']
        self.best_safety_penalty_overall = new_best_obj.get('safety_penalty', INF)
        self.best_diag_penalty_overall = new_best_obj.get('diag_penalty', INF)

    def plot_convergence_curve(self):                                       # MPA.py:459-464 (plotting: out of scope)
        try:
            import matplotlib.pyplot as plt
        except Exception:
            print("matplotlib not available; MPA convergence data is in .convergence_curve_data")
            return
        data = [f for f in self.convergence_curve_data if f is not None]
        if data:
            plt.figure(); plt.plot(data); plt.title("MPA Convergence"); plt.xlabel("Iteration"); plt.ylabel("Best Fitness")
            plt.grid(True); plt.show()
        else:
            print("No MPA convergence data to plot.")
