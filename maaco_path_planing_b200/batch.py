"""Batched sweeps over independent maps (BASELINE config 5: "10k independent 256x256 maps x population 1024,
MPA+MAACO, maps sharded across 8 B200").  Maps are independent units, so they are sharded over the ranks with no
data-path collective, and on each GPU a WAVE of same-shape maps is one mpp_map_batch: every colony pass of the
whole wave is four kernel launches (ranking, tours, best tracking, pheromone update with grid.y = map), enqueued
without host synchronisation.  Results are identical to solving each map alone with the same seed.

The eta'**beta / dist-to-target tables depend only on (shape, start, target, parameters), so a wave shares ONE
table computed on the host with libm (bit-identical to the reference), and tau0 of each map is that shared table
with the map's obstacles masked on the device (mpp_maaco_tables)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .gridmap import START_NODE_VAL, TARGET_NODE_VAL

INF = float("inf")


def shard_maps(n_maps, group=None):
    """[lo, hi) of the maps this rank owns."""
    if group is None:
        return 0, n_maps
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    per = (n_maps + world - 1) // world
    return min(n_maps, rank * per), min(n_maps, (rank + 1) * per)


def default_max_cells(rows, cols):
    """Per-ant path capacity of MAACO and MAACOBatch when `max_cells` is not given: tours are a few (rows + cols) cells
    long (MAACO.py:278-302 never backtracks); a best path that does not fit makes the solve repeat with rows * cols."""
    return min(rows * cols, max(1024, 8 * (rows + cols)))


def _grids_u8(grids):
    """[n_maps, rows, cols] cell codes as uint8 (what mpp_map_batch_create takes): values clipped to 0..255 like
    np.clip(int grid), written straight into the byte array (an int64 wave of 128 256x256 maps is 67 MB: the
    intermediate int64 copies cost more host time than the wave's passes cost on the GPU)."""
    g = np.asarray(grids)
    if g.ndim != 3:
        raise ValueError("grids must be [n_maps, rows, cols]")
    if g.dtype == np.uint8:
        return np.ascontiguousarray(g)
    if g.dtype.kind not in "iub":
        g = g.astype(int)                                                     # (the reference indexes int grids)
    g8 = np.empty(g.shape, np.uint8)
    np.clip(g, 0, 255, out=g8, casting="unsafe")
    return g8


class MAACOBatch:
    """M same-shape maps that share start and target, one colony of `num_ants` ants per map, solved together.
    Same parameters as MAACO (MAACO.py:11-14); `seeds` = one Philox seed per map.  `max_cells` works as in MAACO: left
    at its default, solve() repeats the whole wave with rows*cols cells of path capacity when a best path did not fit;
    given explicitly, such a wave raises MppError."""

    def __init__(self, grids, num_ants, num_iterations, alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min, k_h_adaptive,
                 q0_initial, C0_initial_pheromone=0.1, *, seeds=None, device=None, max_cells=None, ants_per_warp=0,
                 reuse=None):
        import torch
        L = _lib.lib()
        g8 = _grids_u8(grids)
        self.n_maps, self.rows, self.cols = g8.shape
        flat = g8.reshape(self.n_maps, -1)
        if not (flat == START_NODE_VAL).any(axis=1).all():
            raise ValueError("MAACO: Start node not found.")                  # MAACO.py:35-36
        if not (flat == TARGET_NODE_VAL).any(axis=1).all():
            raise ValueError("MAACO: Target node not found.")                 # MAACO.py:37-38
        _lib.require_device()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        h = C.c_void_p()
        _lib.check(L.mpp_map_batch_create(g8.ctypes.data_as(C.c_void_p), self.n_maps, self.rows, self.cols,
                                          self.device_index, C.byref(h)), "mpp_map_batch_create")
        self._maps = h
        self.num_ants, self.num_iterations = int(num_ants), int(num_iterations)
        self.alpha, self.rho, self.Q = alpha, rho, Q
        self._params = _lib.MaacoParams(alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min, k_h_adaptive, q0_initial,
                                        C0_initial_pheromone, num_iterations)
        M, R, Cc, N = self.n_maps, self.rows, self.cols, self.num_ants
        n = R * Cc
        TR = (R + 31) // 32
        self._auto_cells = max_cells is None
        if max_cells is None:
            max_cells = default_max_cells(R, Cc)
        self.max_cells = int(max_cells)
        self._apw = int(ants_per_warp)
        if seeds is None:
            seeds = [int.from_bytes(np.random.bytes(8), "little") for _ in range(M)]
        self.seeds = [int(s) & (2 ** 64 - 1) for s in seeds]
        self._ctor = dict(grids=g8, num_ants=num_ants, num_iterations=num_iterations, alpha=alpha, beta=beta, rho=rho, Q=Q,
                          a_turn_coef=a_turn_coef, wh_max=wh_max, wh_min=wh_min, k_h_adaptive=k_h_adaptive,
                          q0_initial=q0_initial, C0_initial_pheromone=C0_initial_pheromone, seeds=self.seeds,
                          device=self.device_index, ants_per_warp=ants_per_warp)
        dev = self.device
        f64, i32, i64, u8 = torch.float64, torch.int32, torch.int64, torch.uint8
        K = max(1, self.num_iterations)
        key = (M, R, Cc, N, self.max_cells, K, self.device_index)
        if reuse is not None and getattr(reuse, "_key", None) == key:
            # the previous wave's device buffers (same shapes): nothing to allocate, only `touched` / counters to clear
            for name in ("_tau", "_E01", "_dist_t", "_rank", "_slabs", "_touched", "_moves", "_result", "_deposit", "_okbits",
                         "_best_cells", "_steps", "_log"):
                setattr(self, name, getattr(reuse, name))
            self._touched.zero_()
            self._steps.zero_()
        else:
            self._tau = torch.empty((M, n), dtype=f64, device=dev)
            self._E01 = torch.empty(2 * n, dtype=f64, device=dev)             # shared by the whole wave
            self._dist_t = torch.empty(n, dtype=f64, device=dev)
            self._rank = torch.empty(M * L.mpp_maaco_rank_words(R, Cc), dtype=i32, device=dev)
            self._slabs = torch.empty(M * L.mpp_maaco_slab_words(TR, Cc, N), dtype=i32, device=dev)
            self._touched = torch.zeros(M * L.mpp_maaco_touched_words(TR, Cc, N), dtype=i32, device=dev)
            self._moves = torch.empty(M * N * self.max_cells, dtype=u8, device=dev)
            self._result = torch.zeros((M, N, 2), dtype=i64, device=dev)
            self._deposit = torch.zeros((M, N), dtype=f64, device=dev)
            self._okbits = torch.zeros((M, (N + 31) // 32), dtype=i32, device=dev)
            self._best_cells = torch.zeros((M, self.max_cells + 1), dtype=i32, device=dev)
            self._steps = torch.zeros(1, dtype=i64, device=dev)
            self._log = torch.zeros((M, K, 4), dtype=f64, device=dev)
        self._key = key
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(L.mpp_maaco_tables(self._maps, C.byref(self._params), _lib.ptr(self._tau), n, _lib.ptr(self._E01),
                                      _lib.ptr(self._dist_t), stream), "mpp_maaco_tables")
        self._seeds = torch.from_numpy(np.array(self.seeds, np.uint64).view(np.int64)).to(dev)
        st = bytes(_lib.MaacoState(INF, -1, 0, 0, -1, INF, -1, -1))
        self._state = torch.frombuffer(bytearray(st * M), dtype=u8).to(dev)
        self._colony = _lib.Colony(
            self._tau.data_ptr(), n, self._E01.data_ptr(), 0, self._rank.data_ptr(), self._slabs.data_ptr(),
            self._touched.data_ptr(), self._moves.data_ptr(), self.max_cells, K, self._result.data_ptr(),
            self._deposit.data_ptr(), self._okbits.data_ptr(), self._state.data_ptr(), self._best_cells.data_ptr(),
            self._log.data_ptr(), self._steps.data_ptr(), self._seeds.data_ptr(), None)
        self._iter_done = 0
        self.kernel_launches = 0

    def close(self):
        h, self._maps = getattr(self, "_maps", None), None
        if h:
            _lib.lib().mpp_map_batch_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run_iteration(self, it):
        """Enqueue one colony pass of every map of the wave (asynchronous)."""
        import torch
        if not 1 <= it <= max(1, self.num_iterations):
            raise ValueError(f"iteration {it} outside 1..{self.num_iterations}")
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(_lib.lib().mpp_maaco_pass(self._maps, C.byref(self._colony), C.byref(self._params), it, self.num_ants,
                                             self._apw, stream), "mpp_maaco_pass")
        self.kernel_launches += 4
        self._iter_done = max(self._iter_done, it)

    def pheromone(self):
        return self._tau.cpu().numpy().reshape(self.n_maps, self.rows, self.cols)

    def last_results(self):
        """(n_cells, length, turns), each [n_maps, num_ants], of the last pass."""
        import torch
        torch.cuda.synchronize(self.device)
        rec = self._result.cpu().numpy().view(np.dtype([("length", "<f8"), ("n_cells", "<i4"), ("turns", "<i4")]))
        rec = rec.reshape(self.n_maps, self.num_ants)
        return rec["n_cells"].copy(), rec["length"].copy(), rec["turns"].copy()

    def total_steps(self):
        return int(self._steps.cpu().item())

    def solve(self):
        """Runs the remaining iterations; returns one (path, length, turns, convergence_curve) per map -- the values
        MAACO.solve_path_planning (MAACO.py:334-371) returns / stores for that map."""
        import torch
        for it in range(self._iter_done + 1, self.num_iterations + 1):
            self.run_iteration(it)
        torch.cuda.synchronize(self.device)
        M, K = self.n_maps, self.num_iterations
        st = np.frombuffer(self._state.cpu().numpy().tobytes(), dtype=np.dtype(
            [("best_len", "<f8"), ("best_turns", "<i4"), ("best_n_cells", "<i4"), ("best_iter", "<i4"), ("best_ant", "<i4"),
             ("iter_best_len", "<f8"), ("iter_best_turns", "<i4"), ("iter_best_ant", "<i4")]))
        if (st["best_n_cells"] - 1 > self.max_cells).any():
            if not self._auto_cells or self.max_cells >= self.rows * self.cols:
                raise _lib.MppError(f"a tour outgrew max_cells={self.max_cells} (best path: "
                                    f"{int(st['best_n_cells'].max())} cells); re-run with a larger max_cells")
            # the solve is a deterministic function of (grids, parameters, seeds): repeat the wave with full path capacity
            again = type(self)(max_cells=self.rows * self.cols, **self._ctor)
            again.kernel_launches = self.kernel_launches
            self.close()
            self.__dict__.update(again.__dict__)
            again._maps = None                                                # the map handle is ours now
            return self.solve()
        best = self._best_cells.cpu().numpy()
        log = self._log.cpu().numpy()[:, :K]
        out = []
        for k in range(M):
            nb = int(st["best_n_cells"][k])
            pr, pc = np.divmod(best[k, :nb], self.cols)
            path = list(zip(pr.tolist(), pc.tolist()))
            turns = int(st["best_turns"][k]) if st["best_turns"][k] >= 0 else INF
            curve = [float(v) if v != INF else None for v in log[k, :, 2]]
            out.append((path, float(st["best_len"][k]), turns, curve))
        return out


def _waves(grids, lo, hi, wave):
    """Group this rank's maps into waves of same shape / start / target (what one mpp_map_batch needs)."""
    groups = {}
    for i in range(lo, hi):
        g = np.asarray(grids[i])
        s, t = np.argwhere(g == START_NODE_VAL), np.argwhere(g == TARGET_NODE_VAL)
        key = (g.shape, tuple(s[0]) if len(s) else None, tuple(t[0]) if len(t) else None)
        groups.setdefault(key, []).append(i)
    for idx in groups.values():
        for w0 in range(0, len(idx), wave):
            yield idx[w0:w0 + wave]


def solve_maaco_batch(grids, num_ants, num_iterations, params, seeds=None, wave=256, group=None, device=None,
                      max_cells=None):
    """Run MAACO on every grid of `grids` (this rank's shard when `group` is given), `wave` maps per launch.

    Returns a list of (map_index, path, length, turns, convergence_curve) for the maps of this rank; results
    are identical to solving each map alone (same seeds => same Philox streams)."""
    lo, hi = shard_maps(len(grids), group)
    out = []
    prev = None
    for idx in _waves(grids, lo, hi, wave):
        b = MAACOBatch(np.stack([np.asarray(grids[i]) for i in idx]), num_ants, num_iterations,
                       seeds=None if seeds is None else [seeds[i] for i in idx], device=device, max_cells=max_cells,
                       reuse=prev, **params)
        for i, (path, length, turns, curve) in zip(idx, b.solve()):
            out.append((i, path, length, turns, curve))
        b.close()
        prev = b
    out.sort(key=lambda r: r[0])
    return out


class MPABatch:
    """M same-shape maps, one MPA population of `num_predators` paths per map, every iteration of every map in one
    launch (mpp_mpa_iteration_batch); the stable sorts (MPA.py:333,412) are a batched device argsort whose index
    the kernel reads through, and the best-so-far cascade (MPA.py:415-437) is a few vector operations over the maps --
    no host round trip inside the solve.  Same parameters as MPA (MPA.py:10-18); `seeds` = one Philox seed per map."""

    def __init__(self, grids, num_predators, num_iterations, FADs_rate=0.2, P_const=0.5, levy_beta=1.5,
                 turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5, allow_diagonal_moves=True,
                 restrict_diagonal_near_obstacle=True, diagonal_obstacle_penalty=1000.0, *, seeds=None, device=None,
                 max_cells=None, heap_cap=None, warps_per_map=None):
        import math
        import torch
        from .engine import make_policy
        L = _lib.lib()
        g8 = _grids_u8(grids)
        self.n_maps, self.rows, self.cols = g8.shape
        flat = g8.reshape(self.n_maps, -1)
        if not (flat == START_NODE_VAL).any(axis=1).all():
            raise ValueError("MPA: Start node not found in grid.")            # MPA.py:36-37
        if not (flat == TARGET_NODE_VAL).any(axis=1).all():
            raise ValueError("MPA: Target node not found in grid.")           # MPA.py:38-39
        _lib.require_device()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self._grids8 = g8
        h = C.c_void_p()
        _lib.check(L.mpp_map_batch_create(self._grids8.ctypes.data_as(C.c_void_p), self.n_maps, self.rows, self.cols,
                                          self.device_index, C.byref(h)), "mpp_map_batch_create")
        self._maps = h
        self.num_predators, self.num_iterations = int(num_predators), int(num_iterations)
        self.FADs_rate, self.P_const, self.levy_beta = FADs_rate, P_const, levy_beta
        self.policy = make_policy(turn_penalty_factor, safety_penalty_factor, min_safe_distance, diagonal_obstacle_penalty,
                                  restrict_diagonal_near_obstacle, allow_diagonal_moves, mode=1)
        b = levy_beta                                                         # Levy sigma MPA.py:251-253
        num = math.gamma(1 + b) * math.sin(math.pi * b / 2)
        den = math.gamma((1 + b) / 2) * b * (2 ** ((b - 1) / 2))
        sig = (num / den) ** (1 / b) if den > 1e-9 else 1.0
        if isinstance(sig, complex):
            raise ValueError("levy_beta gives a complex Levy sigma in the reference expression (MPA.py:253)")
        self._levy_sigma = float(sig)
        n = self.rows * self.cols
        self.max_cells = int(max_cells or min(n, max(1024, 4 * (self.rows + self.cols))))
        self.heap_cap = int(heap_cap or min(8 * n, max(4096, n // 4)))
        if seeds is None:
            seeds = [int.from_bytes(np.random.bytes(8), "little") for _ in range(self.n_maps)]
        self.seeds = [int(s) & (2 ** 64 - 1) for s in seeds]
        sm = torch.cuda.get_device_properties(self.device).multi_processor_count
        # search slots (one warp each): three CTAs of 8 warps per SM in total, split evenly over the maps (at least one CTA each)
        self.warps_per_map = int(warps_per_map or max(8, ((sm * 24) // self.n_maps) // 8 * 8))
        self._ctor = dict(grids=grids, num_predators=num_predators, num_iterations=num_iterations, FADs_rate=FADs_rate,
                          P_const=P_const, levy_beta=levy_beta, turn_penalty_factor=turn_penalty_factor,
                          safety_penalty_factor=safety_penalty_factor, min_safe_distance=min_safe_distance,
                          allow_diagonal_moves=allow_diagonal_moves,
                          restrict_diagonal_near_obstacle=restrict_diagonal_near_obstacle,
                          diagonal_obstacle_penalty=diagonal_obstacle_penalty, seeds=self.seeds, device=device,
                          warps_per_map=warps_per_map)
        self.predator_evaluations = 0
        self.kernel_launches = 0

    def close(self):
        h, self._maps = getattr(self, "_maps", None), None
        if h:
            _lib.lib().mpp_map_batch_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def solve(self):
        """Returns one (path, length, turns, safety_p, diag_p, fitness, convergence_curve) per map -- what
        MPA.solve_path_planning (MPA.py:320-448) returns / stores for that map."""
        import torch
        t = torch
        L = _lib.lib()
        dev = self.device
        M, N, K, mc = self.n_maps, self.num_predators, self.num_iterations, self.max_cells
        words = (self.rows * self.cols + 31) // 32
        slots = self.warps_per_map * M
        slot_bytes = L.mpp_astar_slot_bytes(self.rows, self.cols, self.heap_cap)
        scratch = t.zeros(256 + max(slots, M) * slot_bytes, dtype=t.uint8, device=dev)
        cells = [t.zeros((M, N, mc), dtype=t.int32, device=dev) for _ in range(2)]
        ncell = [t.zeros((M, N), dtype=t.int32, device=dev) for _ in range(2)]
        stats = [t.zeros((M, N, 5), dtype=t.float64, device=dev) for _ in range(2)]
        tmp = t.empty((slots, mc), dtype=t.int32, device=dev)
        avoid = t.empty((slots, words), dtype=t.int32, device=dev)
        queue = t.zeros(M, dtype=t.int32, device=dev)
        status = t.zeros(1, dtype=t.int32, device=dev)
        counters = t.zeros(4, dtype=t.int64, device=dev)
        seeds = t.from_numpy(np.array(self.seeds, np.uint64).view(np.int64)).to(dev)
        stream = C.c_void_p(t.cuda.current_stream(dev).cuda_stream)
        # ---- initial population: one search per map, replicated (MPA.py:231-245) ----
        _lib.check(L.mpp_mpa_init_batch(self._maps, C.byref(self.policy), N, mc, _lib.ptr(cells[0]), _lib.ptr(ncell[0]),
                                        _lib.ptr(stats[0]), _lib.ptr(scratch), scratch.numel(), self.heap_cap,
                                        _lib.ptr(status), _lib.ptr(counters), stream), "mpp_mpa_init_batch")
        cells[0][:, 1:] = cells[0][:, :1]
        ncell[0][:, 1:] = ncell[0][:, :1]
        stats[0][:, 1:] = stats[0][:, :1]
        self.kernel_launches += 1
        rows = t.arange(M, device=dev)

        def elite(buf):
            order = t.sort(stats[buf][:, :, 4], dim=1, stable=True).indices.to(t.int32).contiguous()   # list.sort is stable
            e = order[:, 0].long()
            return order, stats[buf][rows, e], cells[buf][rows, e], ncell[buf][rows, e]

        order, best_stats, best_cells, best_n = elite(0)                       # MPA.py:322-330
        best_stats, best_cells, best_n = best_stats.clone(), best_cells.clone(), best_n.clone()
        curve = t.empty((K + 1, M), dtype=t.float64, device=dev)
        curve[0] = best_stats[:, 4]
        cur = 0
        for it in range(1, K + 1):
            ratio = it / K
            CF = 0.0 if ratio >= 1.0 else ((1.0 - ratio) ** (2.0 * ratio) if ratio > 0 else 1.0)   # MPA.py:336
            phase = 1 if it <= K / 3 else (2 if it <= 2 * K / 3 else 3)
            nxt = cur ^ 1
            _lib.check(L.mpp_mpa_iteration_batch(
                self._maps, C.byref(self.policy), N, it, phase, self.P_const, CF, self.FADs_rate, self._levy_sigma,
                self.levy_beta, _lib.ptr(seeds), _lib.ptr(order), _lib.ptr(cells[cur]), _lib.ptr(ncell[cur]),
                _lib.ptr(stats[cur]), mc, _lib.ptr(cells[nxt]), _lib.ptr(ncell[nxt]), _lib.ptr(stats[nxt]), _lib.ptr(tmp),
                _lib.ptr(avoid), _lib.ptr(scratch), scratch.numel(), self.warps_per_map, self.heap_cap, _lib.ptr(queue),
                _lib.ptr(status), _lib.ptr(counters), stream), "mpp_mpa_iteration_batch")
            self.kernel_launches += 1
            self.predator_evaluations += M * N
            cur = nxt
            order, cs, cc, cn = elite(cur)                                      # sort :412, population[0]
            # best-so-far cascade MPA.py:415-437, for every map at once (columns: length, turns, safety, diag, fitness)
            eq = lambda a, b: (a - b).abs() < 1e-9
            better = cs[:, 4] < best_stats[:, 4]
            tie = eq(cs[:, 4], best_stats[:, 4]) & ~better
            eL, eT, eS = eq(cs[:, 0], best_stats[:, 0]), eq(cs[:, 1], best_stats[:, 1]), eq(cs[:, 2], best_stats[:, 2])
            casc = (cs[:, 0] < best_stats[:, 0]) | (eL & (cs[:, 1] < best_stats[:, 1])) | \
                   (eL & eT & (cs[:, 2] < best_stats[:, 2])) | (eL & eT & eS & (cs[:, 3] < best_stats[:, 3]))
            upd = better | (tie & casc)
            best_stats = t.where(upd[:, None], cs, best_stats)
            best_cells = t.where(upd[:, None], cc, best_cells)
            best_n = t.where(upd, cn, best_n)
            curve[it] = best_stats[:, 4]
        t.cuda.synchronize(dev)
        st = int(status.item())
        if st:                                                                   # a heap or a path buffer overflowed: the solve
            kw = dict(self._ctor)                                                # is deterministic -- repeat it with more room
            if st == 1:
                if self.heap_cap >= 8 * self.rows * self.cols:
                    raise _lib.MppError("A* heap overflow at maximum capacity")
                kw.update(heap_cap=min(8 * self.rows * self.cols, self.heap_cap * 4), max_cells=self.max_cells)
            else:
                if self.max_cells >= 2 * self.rows * self.cols:
                    raise _lib.MppError("path buffer overflow at maximum capacity")
                kw.update(max_cells=min(2 * self.rows * self.cols, 2 * self.max_cells), heap_cap=self.heap_cap)
            again = MPABatch(**kw)
            again.predator_evaluations, again.kernel_launches = self.predator_evaluations, self.kernel_launches
            out = again.solve()
            self.predator_evaluations, self.kernel_launches = again.predator_evaluations, again.kernel_launches
            again.close()
            return out
        self.expansions = int(counters[0].item())
        bs, bc, bn, cv = best_stats.cpu().numpy(), best_cells.cpu().numpy(), best_n.cpu().numpy(), curve.cpu().numpy()
        out = []
        for k in range(M):
            n = int(bn[k])
            path = [(int(c) // self.cols, int(c) % self.cols) for c in bc[k, :n]]
            length = float(bs[k, 0]) if n > 1 else 0
            col = [float(v) if v != INF else None for v in cv[:, k]]
            out.append((path, length, int(bs[k, 1]), float(bs[k, 2]), float(bs[k, 3]), float(bs[k, 4]), col))
        return out


def solve_mpa_batch(grids, num_predators, num_iterations, params, seeds=None, wave=32, group=None, device=None):
    """MPA over this rank's shard of the maps, `wave` maps per launch (grouped by shape).  Returns
    (map_index, path, length, turns, safety_p, diag_p, fitness, convergence_curve) per map of this rank."""
    lo, hi = shard_maps(len(grids), group)
    out = []
    shapes = {}
    for i in range(lo, hi):
        shapes.setdefault(np.asarray(grids[i]).shape, []).append(i)
    for idx_all in shapes.values():
        for w0 in range(0, len(idx_all), wave):
            idx = idx_all[w0:w0 + wave]
            b = MPABatch(np.stack([np.asarray(grids[i]) for i in idx]), num_predators, num_iterations,
                         seeds=None if seeds is None else [seeds[i] for i in idx], device=device, **params)
            for i, r in zip(idx, b.solve()):
                out.append((i,) + tuple(r))
            b.close()
    out.sort(key=lambda r: r[0])
    return out


# ---- A* / Dijkstra over a batch of maps (astar.py, dijkstra.py) ------------------------------------------------------
# algorithm -> (connector variant, the reference's errors for a map without start / target)
_SEARCH_ALGORITHMS = {
    "astar": (0, "AStar: Start node not found in grid.", "AStar: Target node not found in grid."),      # astar.py:19-20
    "dijkstra": (2, "Dijkstra: Start node not found.", "Dijkstra: Target node not found."),           # dijkstra.py:19-20
}


def _search_algorithm(algorithm):
    if algorithm not in _SEARCH_ALGORITHMS:
        raise ValueError(f"algorithm must be 'astar' or 'dijkstra', not {algorithm!r}")
    return _SEARCH_ALGORITHMS[algorithm]


def _check_endpoints(flat, algorithm):
    """Raises the reference constructor's ValueError for the first map (a row of `flat`, cell codes) that has no start
    or no target -- what a loop of AStarSolver / DijkstraSolver constructors over the maps would raise."""
    _, no_start, no_target = _search_algorithm(algorithm)
    flat = np.asarray(flat)
    has_s = (flat == START_NODE_VAL).any(axis=1)
    has_t = (flat == TARGET_NODE_VAL).any(axis=1)
    bad = np.flatnonzero(~(has_s & has_t))
    if bad.size:
        raise ValueError(no_start if not has_s[bad[0]] else no_target)


def _valid_queries(map_index, src, dst, n_maps, n_cells):
    """Bool tensor: query i names a map of the batch and both its endpoints are cells of that map.  The others get the
    empty result without a search (astar.py:37-39)."""
    if not (map_index.dim() == src.dim() == dst.dim() == 1):
        raise ValueError("map_index, src and dst must be 1-D")
    if not (map_index.numel() == src.numel() == dst.numel()):
        raise ValueError(f"map_index, src and dst differ in length ({map_index.numel()}, {src.numel()}, {dst.numel()})")
    return (map_index >= 0) & (map_index < n_maps) & (src >= 0) & (src < n_cells) & (dst >= 0) & (dst < n_cells)


def _shape_waves(grids, lo, hi, wave=None):
    """Maps lo..hi-1 grouped by shape (one mpp_map_batch each), `wave` maps per group at most (None: all of them)."""
    shapes = {}
    for i in range(lo, hi):
        shapes.setdefault(np.asarray(grids[i]).shape, []).append(i)
    out = []
    for idx in shapes.values():
        step = wave or len(idx)
        out += [idx[w0:w0 + step] for w0 in range(0, len(idx), step)]
    return out


class SearchBatch:
    """M same-shape maps for the deterministic baselines: `search` runs any number of A* / Dijkstra queries, each on
    its own map with its own endpoints and avoid set, in one launch with the statistics of every path fused in
    (mpp_astar_batch_maps); `solve` is AStarSolver(grid).solve() / DijkstraSolver(grid).solve() for every map at once.
    Same parameters and defaults as AStarSolver (astar.py:11-14); start and target may differ from map to map."""

    def __init__(self, grids, turn_penalty_factor=0.1, safety_penalty_factor=0.05, min_safe_distance=1.5,
                 allow_diagonal_moves=True, restrict_diagonal_near_obstacle_policy=True,
                 diagonal_obstacle_penalty_value=1000.0, *, device=None, max_cells=None, heap_cap=None, n_slots=None):
        import torch
        from .engine import make_policy
        L = _lib.lib()
        self._grids8 = _grids_u8(grids)
        self.n_maps, self.rows, self.cols = self._grids8.shape
        _lib.require_device()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        h = C.c_void_p()
        _lib.check(L.mpp_map_batch_create(self._grids8.ctypes.data_as(C.c_void_p), self.n_maps, self.rows, self.cols,
                                          self.device_index, C.byref(h)), "mpp_map_batch_create")
        self._maps = h
        self.allow_diagonal_moves = bool(allow_diagonal_moves)
        self.restrict_corners = bool(restrict_diagonal_near_obstacle_policy)   # astar_strictly_restricts_corners
        self.policy = make_policy(turn_penalty_factor, safety_penalty_factor, min_safe_distance,
                                  diagonal_obstacle_penalty_value, restrict_diagonal_near_obstacle_policy,
                                  allow_diagonal_moves, mode=0)
        self.n = self.rows * self.cols
        self.words = (self.n + 31) // 32
        self.heap_cap = int(heap_cap or min(8 * self.n, max(4096, self.n // 4)))        # SearchEngine's sizes
        self.max_cells = int(max_cells or min(self.n, max(4096, 16 * (self.rows + self.cols))))
        self.max_slots = L.mpp_map_batch_max_slots(h)
        self.n_slots = int(n_slots or self.max_slots)
        self.counters = torch.zeros(4, dtype=torch.int64, device=self.device)  # expansions, relaxations, ring / heap pushes
        self.launches = 0
        self._scratch, self._scratch_key = None, None

    def close(self):
        h, self._maps = getattr(self, "_maps", None), None
        if h:
            _lib.lib().mpp_map_batch_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def expansions(self):
        return int(self.counters[0].item())

    def _i32(self, a):
        import torch
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=torch.int32).contiguous()
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32), device=self.device)

    def _launch(self, variant, mi, src, dst, avoid, longest_first):
        """One mpp_astar_batch_maps launch over the given (valid) queries with the current sizes."""
        import torch as t
        n, mc = mi.numel(), self.max_cells
        slots = max(1, min(self.n_slots, n))
        if self._scratch_key != (slots, self.heap_cap):                   # zero-filled once: search stamps live in it
            nbytes = 256 + slots * _lib.lib().mpp_astar_slot_bytes(self.rows, self.cols, self.heap_cap)
            self._scratch = t.zeros(nbytes, dtype=t.uint8, device=self.device)
            self._scratch_key = (slots, self.heap_cap)
        order = None
        if longest_first and n > slots:
            # a search costs roughly the square of its endpoint distance; the launch ends with its slowest query
            dr = t.div(src, self.cols, rounding_mode="floor") - t.div(dst, self.cols, rounding_mode="floor")
            dc = src % self.cols - dst % self.cols
            order = t.argsort(dr.long() ** 2 + dc.long() ** 2, descending=True).to(t.int32).contiguous()
        cells = t.empty((n, mc), dtype=t.int32, device=self.device)
        ncell = t.empty(n, dtype=t.int32, device=self.device)
        g = t.empty(n, dtype=t.float64, device=self.device)
        stats = t.empty((n, 5), dtype=t.float64, device=self.device)
        stream = C.c_void_p(t.cuda.current_stream(self.device).cuda_stream)
        _lib.check(_lib.lib().mpp_astar_batch_maps(
            self._maps, int(variant), _lib.ptr(mi), _lib.ptr(src), _lib.ptr(dst), _lib.ptr(avoid), n,
            int(self.allow_diagonal_moves), int(self.restrict_corners), C.byref(self.policy), _lib.ptr(cells), mc,
            _lib.ptr(ncell), _lib.ptr(g), _lib.ptr(stats), _lib.ptr(self._scratch), self._scratch.numel(), slots,
            self.heap_cap, _lib.ptr(self.counters), _lib.ptr(order), stream), "mpp_astar_batch_maps")
        self.launches += 1
        return cells, ncell, g, stats

    def search(self, variant, map_index, src, dst, avoid_bits=None, *, longest_first=True):
        """Query i: connector `variant` (0 = astar.py, 1 = MPA.py's private A*, 2 = dijkstra.py) from cell src[i] to
        cell dst[i] of map map_index[i], avoiding the cells set in avoid_bits[i] (n x ceil(rows*cols/32) bitmap words,
        or None).  Returns device tensors (cells [n, max_cells] int32, n_cells [n] int32, g [n] float64 = g of the
        popped target, stats [n, 5] float64 = (length, turns, safety, diag, fitness) of the path).  n_cells = 0: no
        path, or an endpoint / map index outside the batch (not searched).  A heap overflow or a truncated path grows
        the buffers and repeats only those queries (the searches are deterministic)."""
        import torch as t
        from .engine import SearchEngine
        mi, src, dst = self._i32(map_index), self._i32(src), self._i32(dst)
        valid = _valid_queries(mi, src, dst, self.n_maps, self.n)
        n = mi.numel()
        avoid = None
        if avoid_bits is not None:
            if isinstance(avoid_bits, np.ndarray):
                avoid_bits = np.ascontiguousarray(avoid_bits).view(np.int32)
            avoid = t.as_tensor(avoid_bits, device=self.device).contiguous().view(t.int32)   # (uint32 words as int32)
            if avoid.numel() != n * self.words:
                raise ValueError(f"avoid_bits must hold {n} x {self.words} words, not {avoid.numel()}")
            avoid = avoid.reshape(n, self.words).contiguous()
        cells = t.zeros((n, self.max_cells), dtype=t.int32, device=self.device)
        ncell = t.zeros(n, dtype=t.int32, device=self.device)
        g = t.full((n,), INF, dtype=t.float64, device=self.device)
        stats = t.tensor([INF, 0.0, 0.0, 0.0, INF], dtype=t.float64, device=self.device).repeat(n, 1)   # helper.py:104-105
        idx = valid.nonzero().squeeze(1)
        while idx.numel():
            sub = lambda x: None if x is None else x.index_select(0, idx).contiguous()
            c, nc, gg, st = self._launch(variant, sub(mi), sub(src), sub(dst), sub(avoid), longest_first)
            if c.shape[1] > cells.shape[1]:                                  # max_cells grew: widen the earlier rows
                wide = t.zeros((n, c.shape[1]), dtype=t.int32, device=self.device)
                wide[:, :cells.shape[1]] = cells
                cells = wide
            cells[idx, :c.shape[1]] = c
            ncell[idx], g[idx], stats[idx] = nc, gg, st
            bad = (nc < 0) | (nc > c.shape[1])
            if not SearchEngine._grow_from(self, int(nc.min().item()), int(nc.max().item())):
                break
            idx = idx[bad]
        return cells, ncell, g, stats

    def solve(self, algorithm="astar"):
        """One start -> target query per map.  Returns, per map, what AStarSolver(grid, ...).solve() (algorithm
        "astar") or DijkstraSolver(grid, ...).solve() ("dijkstra") returns -- (path, length, turns, safety_p, diag_p,
        fitness) -- followed by the value that solver appends to its convergence_curve (g, or None when the path has
        at most one cell)."""
        variant = _search_algorithm(algorithm)[0]
        flat = self._grids8.reshape(self.n_maps, -1)
        _check_endpoints(flat, algorithm)
        src = (flat == START_NODE_VAL).argmax(axis=1)                      # first row-major 2 / 3 (astar.py:17-18)
        dst = (flat == TARGET_NODE_VAL).argmax(axis=1)
        cells, ncell, g, stats = self.search(variant, np.arange(self.n_maps), src, dst)
        cells, ncell, g, stats = cells.cpu().numpy(), ncell.cpu().numpy(), g.cpu().numpy(), stats.cpu().numpy()
        out = []
        for k in range(self.n_maps):
            n = int(ncell[k])
            if n == 0:
                out.append(([], INF, 0, 0.0, 0.0, INF, None))               # helper.py:104-105
                continue
            r, c = np.divmod(cells[k, :n], self.cols)
            path = list(zip(r.tolist(), c.tolist()))
            st = stats[k]
            out.append((path, float(st[0]) if n > 1 else 0, int(st[1]), float(st[2]), float(st[3]), float(st[4]),
                        float(g[k]) if n > 1 else None))                      # astar.py:70 (path and len(path) > 1)
        return out


def solve_search_batch(grids, algorithm, params, wave=None, group=None, device=None):
    """A* or Dijkstra (algorithm "astar" / "dijkstra") start -> target on every grid of `grids` (this rank's shard when
    `group` is given), grouped by shape, `wave` maps per launch (None: all of a shape).  `params` = SearchBatch's keyword
    arguments.  Returns (map_index, path, length, turns, safety_p, diag_p, fitness, g) per map of this rank, g being the
    convergence-curve value (None for a path of at most one cell)."""
    _search_algorithm(algorithm)
    lo, hi = shard_maps(len(grids), group)
    for i in range(lo, hi):                                                  # before any device work
        _check_endpoints(np.asarray(grids[i]).reshape(1, -1), algorithm)
    out = []
    for idx in _shape_waves(grids, lo, hi, wave):
        b = SearchBatch(np.stack([np.asarray(grids[i]) for i in idx]), device=device, **params)
        for i, r in zip(idx, b.solve(algorithm)):
            out.append((i,) + tuple(r))
        b.close()
    out.sort(key=lambda r: r[0])
    return out
