"""PSOSolver -- drop-in for pso.PSOSolver (pso.py:8-240).  Particles live in HBM as torch tensors;
the velocity/position update (mpp_pso_update_batch) and the A*-connector fitness (mpp_waypoint_fitness_maps) are
sm_100a kernels, launched on the map as a batch of one.  The reference's particle loop is *asynchronous* (a particle sees the gbest already
improved by earlier particles of the same iteration, pso.py:187,190 vs :222-229); this is reproduced
exactly by speculating with the current gbest and re-running only the particles after the first
improver.  RNG: Philox streams of the RNG contract (rng_seed=None -> fresh entropy, like the reference).
"""
from __future__ import annotations

import numpy as np

from . import _lib, rng
from .astar import AStarSolver
from .gridmap import START_NODE_VAL, TARGET_NODE_VAL
from .helper import BasePathfinder
from .maaco import _fresh_seed

INF = float("inf")


class PSOSolver(BasePathfinder):
    def __init__(self, grid, num_iterations, num_particles, num_waypoints_per_particle, w, c1, c2,
                 turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5,
                 allow_diagonal_moves=True, restrict_diagonal_near_obstacle_policy=True,
                 diagonal_obstacle_penalty_value=1000.0, *, rng_seed=None, device=None, verbose=True, group=None):
        g = np.asarray(grid)
        s = np.argwhere(g == START_NODE_VAL)
        t = np.argwhere(g == TARGET_NODE_VAL)
        if not s.size > 0:
            raise ValueError("PSO: Start node not found.")              # pso.py:19
        if not t.size > 0:
            raise ValueError("PSO: Target node not found.")             # pso.py:20
        super().__init__(grid, tuple(s[0]), tuple(t[0]), turn_penalty_factor, safety_penalty_factor,
                         min_safe_distance, allow_diagonal_moves, restrict_diagonal_near_obstacle_policy,
                         diagonal_obstacle_penalty_value, device=device)
        self.num_iterations = num_iterations
        self.num_particles = num_particles
        self.num_waypoints = num_waypoints_per_particle
        self.w, self.c1, self.c2 = w, c1, c2
        self.max_vel = max(1.0, 0.15 * max(self.rows, self.cols))       # pso.py:34
        self.path_connector = AStarSolver(grid=self.grid, turn_penalty_factor=0, safety_penalty_factor=0,
                                          min_safe_distance=0, allow_diagonal_moves=self.allow_diagonal_moves,
                                          restrict_diagonal_near_obstacle_policy=self.restrict_diagonal_near_obstacle_policy,
                                          diagonal_obstacle_penalty_value=0, gridmap=self.map, engine=self.engine)
        self.rng_seed = _fresh_seed() if rng_seed is None else int(rng_seed)
        self._seeds = self.engine.torch.from_numpy(np.array([self.rng_seed & (2 ** 64 - 1)], np.uint64).view(np.int64)
                                                   ).to(self.engine.device)
        self.engine.group = group   # fitness evaluation is sharded over the group's ranks (individuals are independent)
        self.verbose = verbose
        self.gbest_particle_data = {'fitness': INF, 'path': [], 'position': []}
        self.fitness_evaluations = 0
        self._state = None

    # ---- single-individual helpers with the reference's names ---------------------------------
    def _reconstruct_path_from_position(self, position_waypoints_float):    # pso.py:56-94
        if not position_waypoints_float:
            return self.path_connector.solve(self.start_node, self.target_node)[0]
        wp = [(max(0, min(self.rows - 1, int(round(p[0])))), max(0, min(self.cols - 1, int(round(p[1])))))
              for p in position_waypoints_float]
        cells = np.array([[r * self.cols + c for r, c in wp]], np.int32)
        pc, nc, _ = self.engine.waypoint_fitness(cells, self.policy)
        n = int(nc[0])
        return self._nodes(pc[0, :n].cpu().numpy()) if n > 0 else []

    def _initialize_particles(self):                                        # pso.py:97-161
        t = self.engine.torch
        dev = self.engine.device
        N, W = self.num_particles, self.num_waypoints
        max_total = N * 20
        acc_pos, acc_vel, acc_stats, acc_cells, acc_ncell = [], [], [], [], []
        n_acc, attempts = 0, 0
        while n_acc < N and attempts < max_total:
            batch = min(max_total - attempts, max(32, int(1.25 * (N - n_acc)) + 8))
            # the attempts of this batch are generated on the device (mpp_pso_init_batch: same Philox streams as the
            # reference harness, pso.py:50-51,105) and evaluated in one launch
            pos_d = t.empty((batch, W, 2), dtype=t.float64, device=dev)
            vel_d = t.empty((batch, W, 2), dtype=t.float64, device=dev)
            wp = t.empty((batch, W), dtype=t.int32, device=dev)
            offs = t.tensor([attempts], dtype=t.int32, device=dev)
            _lib.check(_lib.lib().mpp_pso_init_batch(self.map.handle, batch, _lib.ptr(offs), W, self.max_vel,
                                                     _lib.ptr(self._seeds), _lib.ptr(pos_d), _lib.ptr(vel_d), _lib.ptr(wp),
                                                     self.engine._stream()), "mpp_pso_init_batch")
            self.fitness_evaluations += batch
            cells, ncell, stats = self.engine.waypoint_fitness(wp, self.policy)
            valid = (ncell > 0).cpu().numpy()
            take = np.flatnonzero(valid)
            room = N - n_acc
            if take.size >= room:
                take = take[:room]
                attempts += int(take[-1]) + 1                                  # the loop stops right after the N-th accept
            else:
                attempts += batch
            if take.size:
                idx = t.as_tensor(take, device=dev)
                acc_pos.append(pos_d[idx]); acc_vel.append(vel_d[idx])
                acc_stats.append(stats[idx]); acc_cells.append(cells[idx]); acc_ncell.append(ncell[idx])
                n_acc += take.size
        self.init_attempts = attempts
        if n_acc == 0:
            # pso.py:128-145: no waypoint chain was valid -> ONE particle built from the direct S->T path, with
            # position = velocity = pbest_position = [[0.0, 0.0]] * W; the padding loop :159-160 then copies it
            path_direct = self._reconstruct_path_from_position([]) if W > 0 else []
            if path_direct and path_direct[0] == self.start_node and path_direct[-1] == self.target_node:
                st = self._calculate_stats_for_path(path_direct)
                row = t.as_tensor(np.array([[r * self.cols + c for r, c in path_direct]], np.int32), device=dev)
                acc_pos.append(t.zeros((1, W, 2), dtype=t.float64, device=dev))
                acc_vel.append(t.zeros((1, W, 2), dtype=t.float64, device=dev))
                acc_stats.append(t.as_tensor(np.array([[float(st[1]), float(st[2]), float(st[3]), float(st[4]),
                                                        float(st[5])]]), device=dev))
                acc_cells.append(row)
                acc_ncell.append(t.as_tensor(np.array([len(path_direct)], np.int32), device=dev))
                n_acc = 1
                print("PSO Warning: Population init failed, used a direct A* path as one particle.")
        if n_acc == 0:                                                          # pso.py:147-157
            print("PSO Error: Could not initialize any valid particles.")
            self.gbest_particle_data = {'fitness': INF, 'path': [], 'position': [], 'length': INF, 'turns': 0,
                                        'safety_penalty': 0, 'diag_penalty': 0}
            return False
        mc = max(c.shape[1] for c in acc_cells)
        pad = lambda c: c if c.shape[1] == mc else t.nn.functional.pad(c, (0, mc - c.shape[1]))
        pos = t.cat(acc_pos); vel = t.cat(acc_vel); stats = t.cat(acc_stats)
        cells = t.cat([pad(c) for c in acc_cells]); ncell = t.cat(acc_ncell)
        # gbest = first strictly-best in acceptance order pso.py:121
        fit = stats[:, 4]
        gi = int(t.argmin(fit).item())
        gi = int((fit == fit[gi]).nonzero()[0].item())
        # padding pso.py:159-160: random.choice(self.particles).copy()
        src = list(range(n_acc))
        while len(src) < N:
            st = rng.Stream(self.rng_seed, rng.CLS_PSO_PAD, 0, len(src), prefetch=2)
            src.append(src[st.below(len(src))])
        if len(src) > n_acc:
            idx = t.as_tensor(src, device=dev)
            pos, vel, stats, cells, ncell = pos[idx], vel[idx], stats[idx], cells[idx], ncell[idx]
        self._state = dict(pos=pos.contiguous(), vel=vel.contiguous(), pbest_pos=pos.clone(), pbest_fit=stats[:, 4].clone(),
                           pbest_stats=stats.clone(), pbest_cells=cells.clone(), pbest_ncell=ncell.clone(),
                           cur_stats=stats.clone(), cur_cells=cells.clone(), cur_ncell=ncell.clone())
        self._set_gbest(pos[gi], cells[gi], int(ncell[gi]), stats[gi].cpu().numpy())
        return True

    def _set_gbest(self, pos_row, cells_row, n, st):
        self._gbest_pos = pos_row.clone().contiguous()
        self.gbest_particle_data = {
            'fitness': float(st[4]), 'path': self._nodes(cells_row[:n].cpu().numpy()),
            'position': [list(map(float, p)) for p in pos_row.cpu().numpy()],
            'length': float(st[0]), 'turns': int(st[1]), 'safety_penalty': float(st[2]), 'diag_penalty': float(st[3])}

    def _store_rows(self, name, lo, rel_idx, cells, ncell):
        """Copy selected rows (relative indices into [lo, ...)) of a path batch into a state buffer."""
        t = self.engine.torch
        S = self._state
        buf = S[name + "_cells"]
        if cells.shape[1] > buf.shape[1]:
            buf = t.nn.functional.pad(buf, (0, cells.shape[1] - buf.shape[1]))
            S[name + "_cells"] = buf
        buf[lo + rel_idx, :cells.shape[1]] = cells[rel_idx]
        S[name + "_ncell"][lo + rel_idx] = ncell[rel_idx]

    def _iterate(self, iteration):                                          # pso.py:179-229
        t = self.engine.torch
        S = self._state
        L = _lib.lib()
        N, W = self.num_particles, self.num_waypoints
        pos0, vel0 = S["pos"].clone(), S["vel"].clone()
        start = 0
        rounds = 0
        while start < N:
            n = N - start
            if rounds:
                S["pos"][start:] = pos0[start:]
                S["vel"][start:] = vel0[start:]
            # particles [start, N) are updated; their waypoint cells are rows [start, N) of wp
            wp = t.empty((N, W), dtype=t.int32, device=S["pos"].device)
            first = t.tensor([start], dtype=t.int32, device=S["pos"].device)
            _lib.check(L.mpp_pso_update_batch(self.map.handle, _lib.ptr(S["pos"]), _lib.ptr(S["vel"]),
                                              _lib.ptr(S["pbest_pos"]), _lib.ptr(self._gbest_pos), N, _lib.ptr(first), W,
                                              self.w, self.c1, self.c2, self.max_vel, _lib.ptr(self._seeds), iteration,
                                              _lib.ptr(wp), self.engine._stream()), "mpp_pso_update_batch")
            cells, ncell, stats = self.engine.waypoint_fitness(wp[start:], self.policy)
            self.fitness_evaluations += n
            rounds += 1
            valid = ncell > 0
            fit = stats[:, 4]
            imp_p = valid & (fit < S["pbest_fit"][start:])                   # pso.py:216
            imp_g = imp_p & (fit < self.gbest_particle_data['fitness'])      # pso.py:222
            hit = imp_g.nonzero()
            q = int(hit[0].item()) if hit.numel() else -1
            end = n if q < 0 else q + 1                                      # particles [start, start+end) are final
            v_idx = valid[:end].nonzero().flatten()
            if v_idx.numel():                                                # pso.py:211-214
                S["cur_stats"][start + v_idx] = stats[v_idx]
                self._store_rows("cur", start, v_idx, cells, ncell)
            p_idx = imp_p[:end].nonzero().flatten()
            if p_idx.numel():                                                # pso.py:217-220
                S["pbest_fit"][start + p_idx] = fit[p_idx]
                S["pbest_pos"][start + p_idx] = S["pos"][start + p_idx]
                S["pbest_stats"][start + p_idx] = stats[p_idx]
                self._store_rows("pbest", start, p_idx, cells, ncell)
            if q >= 0:                                                       # pso.py:223-229
                self._set_gbest(S["pos"][start + q], cells[q], int(ncell[q]), stats[q].cpu().numpy())
            start += end
        self.repair_rounds = getattr(self, "repair_rounds", 0) + rounds - 1

    def solve(self):                                                        # pso.py:163-240
        if self.num_waypoints == 0:
            print("PSO running with 0 waypoints (effectively A*).")
            path = self._reconstruct_path_from_position([])
            stats = self._calculate_stats_for_path(path)
            self.gbest_particle_data = {'path': stats[0], 'fitness': stats[5], 'length': stats[1], 'turns': stats[2],
                                        'safety_penalty': stats[3], 'diag_penalty': stats[4], 'position': []}
            self.convergence_curve.append(stats[5])
            return stats
        if not self._initialize_particles():
            print("PSO: Particle initialization failed completely. Returning empty result.")
            return [], INF, 0, 0.0, 0.0, INF
        self.convergence_curve.append(self.gbest_particle_data['fitness'])
        for iteration in range(self.num_iterations):
            self._iterate(iteration)
            self.convergence_curve.append(self.gbest_particle_data['fitness'])
            if self.verbose and ((iteration + 1) % 10 == 0 or iteration == 0 or iteration == self.num_iterations - 1):
                best = self.gbest_particle_data
                print(f"PSO Iter {iteration+1}/{self.num_iterations}: GBestFit={best['fitness']:.2f} "
                      f"(L:{best.get('length',0):.1f}, T:{best.get('turns',0)}, "
                      f"SP:{best.get('safety_penalty',0):.2f}, DP:{best.get('diag_penalty',0):.2f})")
        res = self.gbest_particle_data
        return (res['path'], res.get('length', INF), res.get('turns', INF), res.get('safety_penalty', INF),
                res.get('diag_penalty', INF), res['fitness'])

    @property
    def particles(self):
        """The reference's list-of-dicts view (pso.py:111-118), materialised from device state."""
        S = self._state
        if S is None:
            return []
        pos, vel, pb = S["pos"].cpu().numpy(), S["vel"].cpu().numpy(), S["pbest_pos"].cpu().numpy()
        cs, ps = S["cur_stats"].cpu().numpy(), S["pbest_stats"].cpu().numpy()
        cc, cn = S["cur_cells"].cpu().numpy(), S["cur_ncell"].cpu().numpy()
        pc, pn = S["pbest_cells"].cpu().numpy(), S["pbest_ncell"].cpu().numpy()
        out = []
        for i in range(self.num_particles):
            d = lambda s: {'l': float(s[0]), 't': int(s[1]), 'sp': float(s[2]), 'dp': float(s[3])}
            out.append({'position': pos[i].tolist(), 'velocity': vel[i].tolist(), 'pbest_position': pb[i].tolist(),
                        'pbest_fitness': float(ps[i, 4]), 'pbest_path': self._nodes(pc[i, :pn[i]]),
                        'pbest_stats': d(ps[i]), 'current_fitness': float(cs[i, 4]),
                        'current_path': self._nodes(cc[i, :cn[i]]), 'current_stats': d(cs[i])})
        return out
