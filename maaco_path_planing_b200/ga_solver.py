"""GASolver -- drop-in for ga_solver.GASolver (ga_solver.py:8-223).  Chromosomes (integer waypoints)
live in HBM; tournament selection, crossover + mutation (mpp_ga_select_batch / mpp_ga_breed_batch) and the
A*-connector fitness (mpp_waypoint_fitness_maps) are sm_100a kernels, launched on the map as a batch of one.  Breeding consumes RNG but evaluation
does not, so a whole generation is bred first and evaluated in one batch (ga_solver.py:186-205)."""
from __future__ import annotations

import numpy as np

from . import _lib, rng
from .astar import AStarSolver
from .gridmap import OBSTACLE, START_NODE_VAL, TARGET_NODE_VAL
from .helper import BasePathfinder
from .maaco import _fresh_seed

INF = float("inf")


class GASolver(BasePathfinder):
    def __init__(self, grid, num_generations, population_size, num_waypoints_per_chromosome, mutation_rate,
                 crossover_rate, tournament_size=3, turn_penalty_factor=0.1, safety_penalty_factor=0.05,
                 min_safe_distance=1.5, allow_diagonal_moves=True, restrict_diagonal_near_obstacle_policy=True,
                 diagonal_obstacle_penalty_value=1000.0, *, rng_seed=None, device=None, verbose=True, group=None):
        g = np.asarray(grid)
        s = np.argwhere(g == START_NODE_VAL)
        t = np.argwhere(g == TARGET_NODE_VAL)
        if not s.size > 0:
            raise ValueError("GA: Start node not found.")               # ga_solver.py:19
        if not t.size > 0:
            raise ValueError("GA: Target node not found.")              # ga_solver.py:20
        super().__init__(grid, tuple(s[0]), tuple(t[0]), turn_penalty_factor, safety_penalty_factor,
                         min_safe_distance, allow_diagonal_moves, restrict_diagonal_near_obstacle_policy,
                         diagonal_obstacle_penalty_value, device=device)
        self.num_generations = num_generations
        self.population_size = population_size
        self.num_waypoints = num_waypoints_per_chromosome
        self.mutation_rate = mutation_rate
        self.crossover_rate = crossover_rate
        self.tournament_size = tournament_size
        self.path_connector = AStarSolver(grid=self.grid, turn_penalty_factor=0, safety_penalty_factor=0,
                                          min_safe_distance=0, allow_diagonal_moves=self.allow_diagonal_moves,
                                          restrict_diagonal_near_obstacle_policy=self.restrict_diagonal_near_obstacle_policy,
                                          diagonal_obstacle_penalty_value=0, gridmap=self.map, engine=self.engine)
        self.rng_seed = _fresh_seed() if rng_seed is None else int(rng_seed)
        self._seeds = self.engine.torch.from_numpy(np.array([self.rng_seed & (2 ** 64 - 1)], np.uint64).view(np.int64)
                                                   ).to(self.engine.device)
        self.engine.group = group   # fitness evaluation is sharded over the group's ranks (individuals are independent)
        self.verbose = verbose
        self.best_solution_overall = {'fitness': INF, 'path': []}
        self.fitness_evaluations = 0
        self._pop = None
        self._fallback = None       # the single direct-path individual of ga_solver.py:111-117 (or the dummy of :123)

    # ---- reference-named single-individual helper ----------------------------------------------
    def _reconstruct_path_from_chromosome(self, chromosome):                # ga_solver.py:58-93
        if not chromosome:
            return self.path_connector.solve(self.start_node, self.target_node)[0]
        cells = np.array([[int(r) * self.cols + int(c) for r, c in chromosome]], np.int32)
        pc, nc, _ = self.engine.waypoint_fitness(cells, self.policy)
        n = int(nc[0])
        return self._nodes(pc[0, :n].cpu().numpy()) if n > 0 else []

    def _evaluate(self, chrom):
        self.fitness_evaluations += chrom.shape[0]
        return self.engine.waypoint_fitness(chrom, self.policy)

    def _initialize_population(self):                                       # ga_solver.py:95-133
        t = self.engine.torch
        dev = self.engine.device
        N, W = self.population_size, self.num_waypoints
        max_total = N * 20
        acc = []
        n_acc, attempts = 0, 0
        while n_acc < N and attempts < max_total:
            batch = min(max_total - attempts, max(32, int(1.25 * (N - n_acc)) + 8))
            chrom_d = t.empty((batch, W), dtype=t.int32, device=dev)             # _create_chromosome :55-56 on the device
            offs = t.tensor([attempts], dtype=t.int32, device=dev)
            _lib.check(_lib.lib().mpp_ga_init_batch(self.map.handle, batch, _lib.ptr(offs), W, _lib.ptr(self._seeds),
                                                    _lib.ptr(chrom_d), self.engine._stream()), "mpp_ga_init_batch")
            cells, ncell, stats = self._evaluate(chrom_d)
            take = np.flatnonzero((ncell > 0).cpu().numpy())
            room = N - n_acc
            if take.size >= room:
                take = take[:room]
                attempts += int(take[-1]) + 1
            else:
                attempts += batch
            if take.size:
                idx = t.as_tensor(take, device=dev)
                acc.append((chrom_d[idx], stats[idx], cells[idx], ncell[idx]))
                n_acc += take.size
        self.init_attempts = attempts
        if n_acc == 0:
            # ga_solver.py:111-117: ONE individual {chromosome: [], path: direct S->T path}; padding :129-130 copies it
            path_direct = self._reconstruct_path_from_chromosome([]) if W > 0 else []
            if path_direct and path_direct[0] == self.start_node and path_direct[-1] == self.target_node:
                st = self._calculate_stats_for_path(path_direct)
                ind = {'chromosome': [], 'path': list(path_direct), 'fitness': float(st[5]), 'length': float(st[1]),
                       'turns': int(st[2]), 'safety_penalty': float(st[3]), 'diag_penalty': float(st[4])}
                print("GA Warning: Population init failed, used a direct A* path as one individual.")
                # Every later generation reproduces this individual: crossover of two empty chromosomes is empty
                # (:144-152), _mutate returns [] (:155), and the child's path is the same direct path -- so the
                # population is a fixed point and no kernel has anything to evaluate.
                self._fallback = ind
                return True
            print("GA Error: Could not initialize any valid individuals.")            # :120-126
            self._fallback = {'chromosome': [], 'path': [], 'fitness': INF, 'length': INF, 'turns': 0,
                              'safety_penalty': 0, 'diag_penalty': 0}
            self._fallback_failed = True
            return False
        mc = max(a[2].shape[1] for a in acc)
        pad = lambda c: c if c.shape[1] == mc else t.nn.functional.pad(c, (0, mc - c.shape[1]))
        chrom = t.cat([a[0] for a in acc]); stats = t.cat([a[1] for a in acc])
        cells = t.cat([pad(a[2]) for a in acc]); ncell = t.cat([a[3] for a in acc])
        src = list(range(n_acc))
        while len(src) < N:                                                 # padding :129-130
            st = rng.Stream(self.rng_seed, rng.CLS_GA_PAD, 0, len(src), prefetch=2)
            src.append(src[st.below(len(src))])
        if len(src) > n_acc:
            idx = t.as_tensor(src, device=dev)
            chrom, stats, cells, ncell = chrom[idx], stats[idx], cells[idx], ncell[idx]
        self._set_population(chrom, stats, cells, ncell)                    # sort :132
        return True

    def _set_population(self, chrom, stats, cells, ncell):
        t = self.engine.torch
        order = t.sort(stats[:, 4], stable=True).indices                    # list.sort is stable
        self._pop = dict(chrom=chrom[order].contiguous(), stats=stats[order].contiguous(),
                         cells=cells[order], ncell=ncell[order])

    def _individual(self, i):
        P = self._pop
        st = P["stats"][i].cpu().numpy()
        n = int(P["ncell"][i])
        return {'chromosome': self._nodes(P["chrom"][i].cpu().numpy()), 'path': self._nodes(P["cells"][i, :n].cpu().numpy()),
                'fitness': float(st[4]), 'length': float(st[0]), 'turns': int(st[1]), 'safety_penalty': float(st[2]),
                'diag_penalty': float(st[3])}

    @property
    def population(self):
        if self._fallback is not None:
            return [dict(self._fallback) for _ in range(self.population_size)]
        return [] if self._pop is None else [self._individual(i) for i in range(self.population_size)]

    def _generation(self, gen):                                             # ga_solver.py:178-209
        t = self.engine.torch
        L = _lib.lib()
        P = self._pop
        N, W = self.population_size, self.num_waypoints
        dev = self.engine.device
        parents = t.empty(N, dtype=t.int32, device=dev)
        fit = P["stats"][:, 4].contiguous()
        _lib.check(L.mpp_ga_select_batch(self.map.handle, _lib.ptr(fit), N, self.tournament_size, _lib.ptr(self._seeds),
                                         gen, _lib.ptr(parents), self.engine._stream()), "mpp_ga_select_batch")
        children = t.empty((N, W), dtype=t.int32, device=dev)
        _lib.check(L.mpp_ga_breed_batch(self.map.handle, _lib.ptr(P["chrom"]), _lib.ptr(parents), N, W,
                                        self.crossover_rate, self.mutation_rate, _lib.ptr(self._seeds), gen,
                                        _lib.ptr(children), self.engine._stream()), "mpp_ga_breed_batch")
        cells, ncell, stats = self._evaluate(children)
        # invalid child -> the parent object: p1 for even slots, p2 for odd (:204-205)
        bad = (ncell <= 0).nonzero().flatten()
        if bad.numel():
            slot = bad
            pidx = parents[((slot // 2) * 2 + (slot % 2)) % N].long()
            if P["cells"].shape[1] > cells.shape[1]:
                cells = t.nn.functional.pad(cells, (0, P["cells"].shape[1] - cells.shape[1]))
            k = min(cells.shape[1], P["cells"].shape[1])
            children[slot] = P["chrom"][pidx]
            stats[slot] = P["stats"][pidx]
            cells[slot, :k] = P["cells"][pidx, :k]
            ncell[slot] = P["ncell"][pidx]
        self._set_population(children, stats, cells, ncell)                 # :208-209

    def solve(self):                                                        # ga_solver.py:162-223
        if self.num_waypoints == 0:
            print("GA running with 0 waypoints (effectively A*).")
            path = self._reconstruct_path_from_chromosome([])
            stats = self._calculate_stats_for_path(path)
            self.best_solution_overall = {'path': stats[0], 'fitness': stats[5], 'length': stats[1], 'turns': stats[2],
                                          'safety_penalty': stats[3], 'diag_penalty': stats[4]}
            self.convergence_curve.append(stats[5])
            return stats
        if not self._initialize_population():
            print("GA: Population initialization failed completely. Returning empty result.")
            return [], INF, 0, 0.0, 0.0, INF
        self.best_solution_overall = dict(self._fallback) if self._fallback is not None else self._individual(0)
        self.convergence_curve.append(self.best_solution_overall['fitness'])
        for gen in range(self.num_generations):
            if self._fallback is None:
                self._generation(gen)
                if float(self._pop["stats"][0, 4]) < self.best_solution_overall['fitness']:    # :211-213
                    self.best_solution_overall = self._individual(0)
            self.convergence_curve.append(self.best_solution_overall['fitness'])
            if self.verbose and ((gen + 1) % 10 == 0 or gen == 0 or gen == self.num_generations - 1):
                b = self.best_solution_overall
                print(f"GA Gen {gen+1}/{self.num_generations}: BestFit={b['fitness']:.2f} "
                      f"(L:{b['length']:.1f}, T:{b['turns']}, SP:{b['safety_penalty']:.2f}, DP:{b['diag_penalty']:.2f})")
        res = self.best_solution_overall
        return (res['path'], res['length'], res['turns'], res['safety_penalty'], res['diag_penalty'], res['fitness'])
