"""MAACO -- drop-in for the reference class ``MAACO.MAACO`` (MAACO.py:10-377) whose colony pass
(tour construction, best tracking, pheromone update) runs as sm_100a kernels behind the C ABI.

Same constructor arguments, attributes and return values as the reference; additive keyword-only
arguments select the RNG stream seed, the device and the (optional) ``torch.distributed`` group
over which the colony is sharded.  No CPU fallback: without libmpp_b200.so or a B200 this raises.

Keyword-only additions (none changes a result; every combination is bit-identical, see tests/test_maaco_gpu.py):
  rng_seed        seed of the Philox streams (DESIGN.md section 2); None = from os.urandom (or $MPP_RNG_SEED)
  device, group   CUDA device index; torch.distributed group to shard the colony over
  ants_per_warp   form of the tour kernel (one thread per ant): 0 = chosen from the colony size, or 1, 2, 4, ..., 32
  max_cells       capacity of the per-ant tour buffers (default 8*(rows+cols); the solve repeats itself with rows*cols
                  if the best path did not fit; a colony sharded over the all-gather exchange grows them instead when
                  any tour does not fit)
"""
from __future__ import annotations

import ctypes as C
import math
import os

import numpy as np

from . import _lib
from . import dist as dist_mod
from .batch import default_max_cells
from .dist import padded_tile_rows
from .gridmap import GridMap, START_NODE_VAL, TARGET_NODE_VAL

INF = float("inf")


def _round64k(x):
    return ((int(x) + 65535) // 65536) * 65536


def _fresh_seed():
    """Seed of a solver built without rng_seed=: fresh entropy, like the reference's never-seeded RNGs -- unless
    MPP_RNG_SEED is set, which makes unmodified callers (the reference's main.py) reproducible."""
    env = os.environ.get("MPP_RNG_SEED")
    if env:
        return int(env, 0)
    return int.from_bytes(os.urandom(8), "little")


class MAACO:
    def __init__(self, grid, num_ants, num_iterations,
                 alpha, beta, rho, Q,
                 a_turn_coef, wh_max, wh_min, k_h_adaptive, q0_initial,
                 C0_initial_pheromone=0.1, *,
                 rng_seed=None, device=None, max_cells=None, ants_per_warp=0, group=None, verbose=True):
        import torch
        self._ctor = dict(grid=grid, num_ants=num_ants, num_iterations=num_iterations, alpha=alpha, beta=beta, rho=rho,
                          Q=Q, a_turn_coef=a_turn_coef, wh_max=wh_max, wh_min=wh_min, k_h_adaptive=k_h_adaptive,
                          q0_initial=q0_initial, C0_initial_pheromone=C0_initial_pheromone, rng_seed=rng_seed,
                          device=device, ants_per_warp=ants_per_warp, group=group, verbose=verbose)
        self.grid = np.array(grid, dtype=int)                       # MAACO.py:15
        self.rows, self.cols = self.grid.shape
        self.num_ants = num_ants
        self.num_iterations = num_iterations
        self.alpha, self.beta, self.rho, self.Q = alpha, beta, rho, Q
        self.a_turn_coef, self.wh_max, self.wh_min = a_turn_coef, wh_max, wh_min
        self.k_h_adaptive, self.q0_initial = k_h_adaptive, q0_initial
        self.k0_iter_threshold_factor = 0.7
        self.C0_base = C0_initial_pheromone
        s = np.argwhere(self.grid == START_NODE_VAL)
        t = np.argwhere(self.grid == TARGET_NODE_VAL)
        if not s.size > 0:
            raise ValueError("MAACO: Start node not found.")       # MAACO.py:35-36
        if not t.size > 0:
            raise ValueError("MAACO: Target node not found.")      # MAACO.py:37-38
        self.start_node = (int(s[0][0]), int(s[0][1]))
        self.target_node = (int(t[0][0]), int(t[0][1]))
        d = math.sqrt((self.start_node[0] - self.target_node[0]) ** 2 + (self.start_node[1] - self.target_node[1]) ** 2)
        self.dist_S_to_T_overall = d if d >= 1e-9 else 1e-9
        self.rng_seed = _fresh_seed() if rng_seed is None else int(rng_seed)
        self._ctor["rng_seed"] = self.rng_seed
        self.verbose = verbose
        if ants_per_warp not in (0, 1, 2, 4, 8, 16, 32):
            raise ValueError("ants_per_warp must be 0 (automatic) or a power of two <= 32")
        self._apw = int(ants_per_warp)

        # ---- sharding of the colony over the process group (ants are independent given tau) ----
        self.group = group
        if group is not None:
            import torch.distributed as dist
            self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        else:
            self.world, self.rank = 1, 0
        if num_ants % self.world:
            raise ValueError("num_ants must be divisible by the group size")
        self.n_local = num_ants // self.world
        self.ant_offset = self.rank * self.n_local

        L = _lib.lib()
        self.map = GridMap(self.grid, device=device)
        self._maps = self.map.handle
        self.device = torch.device("cuda", self.map.device)
        n = self.rows * self.cols
        R, Cc = self.rows, self.cols
        self.tile_rows, self.tile_cols = (R + 31) // 32, (Cc + 31) // 32
        # a sharded colony updates tau by slices of whole tile rows (32 cell rows), padded to split evenly
        self.tile_rows_per_rank = padded_tile_rows(self.tile_rows, self.world) // self.world
        npad = self.tile_rows_per_rank * self.world * 32 * Cc
        # per-ant path capacity: tours are a few (R+C) cells long (no backtracking, MAACO.py:278-302); a tour that
        # outgrows the buffer is still constructed and counted exactly -- only its move list is truncated -- and
        # solve_path_planning() re-runs the (deterministic) solve with full capacity if the best path was cut
        self._auto_cells = max_cells is None
        if max_cells is None:
            max_cells = default_max_cells(R, Cc)
        self.max_cells = int(max_cells)
        self.max_cells_hint = self.max_cells                          # what was asked (max_cells can grow, see _rewind)
        dev = self.device
        f64, i32, i64, u8 = torch.float64, torch.int32, torch.int64, torch.uint8
        nl = self.n_local
        self._p2p = None
        if 1 < self.world <= L.mpp_maaco_max_peers() and os.environ.get("MPP_P2P", "1") != "0":
            self._p2p = self._setup_peer_memory(npad)                # NVLink peer memory for the two exchanges (or None)
        if self._p2p is not None:
            self._tau = self._p2p["tau"]
            self._tau.zero_()
        else:
            self._tau = torch.zeros(npad, dtype=f64, device=dev)    # padded so tau slices all-gather evenly
        self._E01 = torch.empty(2 * n, dtype=f64, device=dev)       # eta'**beta, interleaved by turn flag
        self._dist_t = torch.empty(n, dtype=f64, device=dev)
        self._rank = torch.empty(L.mpp_maaco_rank_words(R, Cc), dtype=i32, device=dev)
        self._params = _lib.MaacoParams(alpha, beta, rho, Q, a_turn_coef, wh_max, wh_min, k_h_adaptive, q0_initial,
                                        C0_initial_pheromone, num_iterations)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(L.mpp_maaco_tables(self._maps, C.byref(self._params), _lib.ptr(self._tau), npad, _lib.ptr(self._E01),
                                      _lib.ptr(self._dist_t), C.c_void_p(stream)), "mpp_maaco_tables")
        # visited sets of the local ants as per-tile slabs + the (tile, ant) bitmaps (csrc/mpp_maaco.cu, header comment)
        self._slabs = torch.empty(L.mpp_maaco_slab_words(self.tile_rows, Cc, nl), dtype=i32, device=dev)
        self._touched = torch.zeros(L.mpp_maaco_touched_words(self.tile_rows, Cc, nl), dtype=i32, device=dev)
        self._moves = torch.zeros(nl * self.max_cells, dtype=u8, device=dev)
        if self._p2p is not None:
            self._result = self._p2p["result"]
            self._result.zero_()
        else:
            self._result = torch.zeros((num_ants, 2), dtype=i64, device=dev)   # mpp_ant_result per global ant
        self._deposit = torch.zeros(num_ants, dtype=f64, device=dev)
        self._okbits = torch.zeros((num_ants + 31) // 32, dtype=i32, device=dev)
        self._best_cells = torch.zeros(self.max_cells + 1, dtype=i32, device=dev)
        self._steps = torch.zeros(1, dtype=i64, device=dev)
        self._log = torch.zeros(max(1, num_iterations) * 4, dtype=f64, device=dev)
        self._seeds = torch.from_numpy(np.array([self.rng_seed & (2 ** 64 - 1)], np.uint64).view(np.int64)).to(dev)
        st = _lib.MaacoState(INF, -1, 0, 0, -1, INF, -1, -1)
        self._state = torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).to(dev)
        self._latch = None
        if self.world > 1:
            tr = self.tile_rows_per_rank
            if self._p2p is not None:
                self._slabs_recv, self._touched_recv = self._p2p["slabs"], self._p2p["touched"]
                self._touched_recv.zero_()                           # (slabs need no clearing: valid = touched bit)
            else:
                self._slabs_recv = torch.zeros(L.mpp_maaco_slab_words(tr, Cc, num_ants), dtype=i32, device=dev)
                self._touched_recv = torch.zeros(L.mpp_maaco_touched_words(tr, Cc, num_ants), dtype=i32, device=dev)
            self._latch = torch.zeros(1, dtype=i32, device=dev)
            self._offsets_local = torch.zeros(nl, dtype=i32, device=dev)
            self._offsets = torch.zeros(num_ants, dtype=i32, device=dev)
            self._xhdr = int(L.mpp_maaco_xhdr_bytes(nl))
            # capacity of the move-code area of one rank's exchange buffer: generous for the first two passes, then
            # 1.5 x the largest segment seen two passes earlier (identical on every rank: the totals travel in the
            # headers); an overflow raises the device latch and the pass is repeated with more room
            self._cap_max = _round64k(nl * min(self.max_cells, max(64, 2 * (R + Cc))))
            self._cap = self._cap_max
            if self._p2p is None:
                self._xbuf_local = torch.zeros(self._xhdr + self._cap_max, dtype=u8, device=dev)
                self._xbuf_all = torch.zeros(self.world * (self._xhdr + self._cap_max), dtype=u8, device=dev)
            self._ring = [torch.zeros(self.world + 1, dtype=i32).pin_memory() for _ in range(4)]
            self._ring_ev = [None] * 4
            self._ring_cap = [0] * 4
            self._enqueued = []                                  # (iteration, cap) of passes not yet confirmed
        self._colony = _lib.Colony(
            self._tau.data_ptr(), npad, self._E01.data_ptr(), 0, self._rank.data_ptr(), self._slabs.data_ptr(),
            self._touched.data_ptr(), self._moves.data_ptr(), self.max_cells, max(1, num_iterations),
            self._result.data_ptr(), self._deposit.data_ptr(), self._okbits.data_ptr(), self._state.data_ptr(),
            self._best_cells.data_ptr(), self._log.data_ptr(), self._steps.data_ptr(), self._seeds.data_ptr(),
            self._latch.data_ptr() if self._latch is not None else None)

        if self._p2p is not None:
            # the peers write into this rank's buffers from their very first tour kernel: nobody starts before every rank
            # has cleared them
            import torch.distributed as dist
            torch.cuda.synchronize(dev)
            dist.barrier(group=self.group)
        self.best_path_overall = []
        self.best_path_length_overall = INF
        self.best_path_turns_overall = INF
        self.convergence_curve_data = []
        self._iter_done = 0
        self.kernel_launches = 0

    def _setup_peer_memory(self, npad):
        """Symmetric (peer-mapped) allocations for the sharded colony's two exchanges: every rank's receive buffers of the
        visited slabs and of the results, and every rank's pheromone field, each addressable from all ranks over NVLink.
        Then the producers write straight into the peers (mpp_maaco_tours_p2p / mpp_maaco_pheromone with peer pointers)
        and a pass needs two device-side barriers: no pack, no all-gather, no replay.  Returns None when the platform
        cannot map peer memory (the NCCL all-gathers of move codes and tau slices are then used; same results)."""
        import torch
        import torch.distributed as dist
        ok = 1
        out = None
        try:
            import torch.distributed._symmetric_memory as symm
            L = _lib.lib()
            Cc, tr, N = self.cols, self.tile_rows_per_rank, self.num_ants
            # what the peers write into: this rank's slice of every ant's visited slabs + the (tile, ant) bitmaps, the
            # result table, and the pheromone field
            slabs = symm.empty(int(L.mpp_maaco_slab_words(tr, Cc, N)), dtype=torch.int32, device=self.device)
            touched = symm.empty(int(L.mpp_maaco_touched_words(tr, Cc, N)), dtype=torch.int32, device=self.device)
            result = symm.empty((N, 2), dtype=torch.int64, device=self.device)
            tau = symm.empty(npad, dtype=torch.float64, device=self.device)
            hs = symm.rendezvous(slabs, self.group)
            hb = symm.rendezvous(touched, self.group)
            hr = symm.rendezvous(result, self.group)
            ht = symm.rendezvous(tau, self.group)
            ptrs = lambda h: torch.tensor([int(p) for p in h.buffer_ptrs], dtype=torch.int64, device=self.device)
            harr = lambda h: (C.c_void_p * self.world)(*[int(p) for p in h.buffer_ptrs])   # host arrays (kernel parameters)
            out = dict(slabs=slabs, touched=touched, result=result, tau=tau, hx=hs, ht=ht, hb=hb, hr=hr,
                       speers=harr(hs), bpeers=harr(hb), rpeers=harr(hr), tpeers=ptrs(ht))
        except Exception as e:                                       # noqa: BLE001 -- any failure = no peer memory here
            ok = 0
            self._p2p_error = f"{type(e).__name__}: {e}"
        flag = torch.tensor([ok], dtype=torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)   # all ranks or none
        return out if int(flag.item()) == 1 else None

    # ---- reference attributes materialised from device state ------------------------------
    @property
    def pheromone_matrix(self):
        self._settle()
        n = self.rows * self.cols
        return self._tau[:n].cpu().numpy().reshape(self.rows, self.cols)

    @property
    def dist_to_target_matrix(self):
        return self._dist_t.cpu().numpy().reshape(self.rows, self.cols)

    def _calculate_adaptive_q0(self, current_iteration_num):
        return _lib.lib().mpp_maaco_q0(self.num_iterations, int(current_iteration_num), self.q0_initial)

    # ---- one colony pass (MAACO.py:336-359), fully asynchronous ----------------------------
    def _enqueue_iteration(self, it, events=None):
        """One colony pass.  `events`: optional CUDA events recorded at (start, after tours, before the
        pheromone update, end[, after the ranking kernel]) on the launching stream -- used by bench.py for
        per-kernel timing."""
        import torch
        if not 1 <= it <= max(1, self.num_iterations):               # the per-iteration log has num_iterations rows
            raise ValueError(f"iteration {it} outside 1..{self.num_iterations}")
        if self.world > 1:
            self._confirm(upto=it - 2)                                # lagged, deterministic sizing of the exchange
        self._enqueue_pass(it, events)

    def _enqueue_pass(self, it, events=None):
        import torch
        L = _lib.lib()
        cur = torch.cuda.current_stream(self.device)
        stream = C.c_void_p(cur.cuda_stream)
        col = C.byref(self._colony)
        nl, off, N = self.n_local, self.ant_offset, self.num_ants
        plog = getattr(self, "_phase_log", None)                      # tools/shard_time.py: [(phase, event)] per pass

        def mark(name):
            if plog is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(cur)
                plog.append((name, ev))
        mark("start")
        if events:
            events[0].record(cur)
        _lib.check(L.mpp_maaco_rank(self._maps, col, self.alpha, stream), "mpp_maaco_rank")
        mark("rank")
        if events and len(events) > 4:
            events[4].record(cur)
        p2p = self._p2p if self.world > 1 else None
        if p2p is not None:
            # sharded over peer memory: the tour kernel itself delivers every slab to the rank that updates its tile row
            # and every result to every rank (NVLink stores from the producing kernel)
            _lib.check(L.mpp_maaco_tours_p2p(self._maps, col, it, self._calculate_adaptive_q0(it), self.alpha, nl, off, N,
                                             self._apw, p2p["speers"], p2p["bpeers"], p2p["rpeers"], self.world,
                                             self.tile_rows_per_rank, stream),
                       "mpp_maaco_tours_p2p")
        else:
            _lib.check(L.mpp_maaco_tours(self._maps, col, it, self._calculate_adaptive_q0(it), self.alpha, nl, off, N,
                                         self._apw, stream), "mpp_maaco_tours")
        mark("tours")
        if events:
            events[1].record(cur)
        if self.world == 1:
            _lib.check(L.mpp_maaco_best(self._maps, col, 0, nl, N, self.Q, it, stream), "mpp_maaco_best")
            if events:
                events[2].record(cur)
            _lib.check(L.mpp_maaco_pheromone(self._maps, col, _lib.ptr(self._slabs), _lib.ptr(self._touched), N, 0,
                                             self.tile_rows, self.rho, it, 0, None, 0, stream), "mpp_maaco_pheromone")
            self.kernel_launches += 4
        elif p2p is not None:
            tr = self.tile_rows_per_rank
            p2p["hx"].barrier(channel=0)                               # every rank's tours are done: slabs and results have landed
            mark("exchange")
            # (the local bitmaps of the next pass: the local update never runs on them, so nobody else clears them)
            self._touched.view(2, -1)[(it + 1) & 1].zero_()
            _lib.check(L.mpp_maaco_best(self._maps, col, off, nl, N, self.Q, it, stream), "mpp_maaco_best")
            mark("best")
            if events:
                events[2].record(cur)
            _lib.check(L.mpp_maaco_pheromone(self._maps, col, _lib.ptr(self._slabs_recv), _lib.ptr(self._touched_recv),
                                             N, self.rank * tr, tr, self.rho, it, 0, _lib.ptr(p2p["tpeers"]), self.world,
                                             stream), "mpp_maaco_pheromone")
            mark("pheromone")
            p2p["ht"].barrier(channel=0)                               # every rank's slice has landed in every field
            mark("tau exchange")
            self.kernel_launches += 4
        else:
            cap = self._cap
            seg = self._xhdr + cap
            _lib.check(L.mpp_maaco_xpack(self._maps, col, off, nl, N, _lib.ptr(self._offsets_local),
                                         _lib.ptr(self._xbuf_local), cap, None, self.world, self.rank, stream),
                       "mpp_maaco_xpack")
            mark("xpack")
            # ONE all-gather per pass carries the results and the tours (move codes) of every rank
            dist_mod.exchange_buffers(self._xbuf_all[:self.world * seg], self._xbuf_local[:seg], self.group)
            mark("exchange")
            tr = self.tile_rows_per_rank
            _lib.check(L.mpp_maaco_xunpack(self._maps, col, _lib.ptr(self._xbuf_all), cap, self.world, nl, it,
                                           _lib.ptr(self._offsets), self.rank * tr, tr, _lib.ptr(self._slabs_recv),
                                           _lib.ptr(self._touched_recv), _lib.ptr(self._touched), stream),
                       "mpp_maaco_xunpack")
            mark("xunpack")
            _lib.check(L.mpp_maaco_best(self._maps, col, off, nl, N, self.Q, it, stream), "mpp_maaco_best")
            mark("best")
            if events:
                events[2].record(cur)
            _lib.check(L.mpp_maaco_pheromone(self._maps, col, _lib.ptr(self._slabs_recv), _lib.ptr(self._touched_recv),
                                             N, self.rank * tr, tr, self.rho, it, 1, None, self.world, stream),
                       "mpp_maaco_pheromone")
            mark("pheromone")
            sl = tr * 32 * self.cols
            dist_mod.gather_tau(self._tau, self._tau[self.rank * sl:(self.rank + 1) * sl], self.group)
            mark("tau exchange")
            # what the host needs two passes later: every segment's code total (from the gathered headers) + the latch
            slot = it & 3
            hdr_tot = self._xbuf_all.view(torch.int32).as_strided((self.world,), (seg // 4,), (16 * nl) // 4)
            self._ring[slot][:self.world].copy_(hdr_tot, non_blocking=True)
            self._ring[slot][self.world:].copy_(self._latch, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(cur)
            self._ring_ev[slot] = ev
            self._enqueued.append((it, cap))
            self.kernel_launches += 8
        if events:
            events[3].record(cur)

    def _confirm(self, upto):
        """Sharded colony: wait for the (tiny, asynchronous) header copies of every enqueued pass <= `upto`, size the
        next exchange from them and repeat passes from the first one whose exchange overflowed."""
        while self._enqueued and self._enqueued[0][0] <= upto:
            it, cap = self._enqueued[0]
            slot = it & 3
            self._ring_ev[slot].synchronize()
            vals = self._ring[slot].tolist()
            totals, latch = vals[:self.world], vals[self.world]
            if latch != 0:
                self._rewind(latch, totals)
                continue
            self._enqueued.pop(0)
            self._cap = min(self._cap_max, _round64k(int(1.5 * max(totals)) + 4096))

    def _rewind(self, first_bad, totals):
        """The exchange of pass `first_bad` did not fit: a rank's move codes outgrew the capacity of the exchange (`totals`:
        every rank's code bytes in that pass, from its ring slot) or a tour outgrew max_cells (its codes were cut at the
        source, so no rank could replay it).  Since then every kernel was a no-op (device latch), so the colony is exactly
        as pass first_bad - 1 left it.  Make room and enqueue those passes again."""
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize(self.device)
        redo = [it for it, _ in self._enqueued if it >= first_bad]
        cap_bad = dict(self._enqueued)[first_bad]
        # the longest tour of the bad pass: this rank's own records are still the ones its tour kernel wrote then (the
        # unpack of the other ranks' records may have stopped at the latch)
        own = self._result.view(torch.int32).view(self.num_ants, 4)[self.ant_offset:self.ant_offset + self.n_local, 2]
        longest = (own.max() - 1).reshape(1)
        dist.all_reduce(longest, op=dist.ReduceOp.MAX, group=self.group)
        longest = int(longest.item())
        if max(totals) <= cap_bad and longest <= self.max_cells:
            raise _lib.MppError(f"sharded colony: the exchange of pass {first_bad} was stopped without an overflow")
        if longest > self.max_cells:
            self._grow_moves(min(self.rows * self.cols, max(longest, 2 * self.max_cells)))
        if max(totals) > cap_bad:
            self._cap_max = max(self._cap_max, _round64k(2 * max(totals)))
        self._cap = self._cap_max
        if self._xbuf_local.numel() < self._xhdr + self._cap_max:
            self._xbuf_local = torch.zeros(self._xhdr + self._cap_max, dtype=torch.uint8, device=self.device)
            self._xbuf_all = torch.zeros(self.world * (self._xhdr + self._cap_max), dtype=torch.uint8, device=self.device)
        self._latch.zero_()
        # the tours of the bad pass DID run (the latch rises behind them): their (tile, ant) bits must not be there when the
        # pass is repeated, or a window slide would reload the first attempt's slab -- the ant's own future cells -- as visited
        self._touched.zero_()
        self._enqueued = [e for e in self._enqueued if e[0] < first_bad]
        self.exchange_rewinds = getattr(self, "exchange_rewinds", 0) + 1
        for it in redo:
            self._enqueue_pass(it)

    def _grow_moves(self, max_cells):
        """Per-ant move buffers (and the best path) of `max_cells` moves; the best path found so far is kept."""
        import torch
        best = self._best_cells
        self.max_cells = int(max_cells)
        self._moves = torch.zeros(self.n_local * self.max_cells, dtype=torch.uint8, device=self.device)
        self._best_cells = torch.zeros(self.max_cells + 1, dtype=torch.int32, device=self.device)
        self._best_cells[:best.numel()].copy_(best)
        self._colony.moves, self._colony.best_cells = self._moves.data_ptr(), self._best_cells.data_ptr()
        self._colony.max_cells = self.max_cells

    def _settle(self):
        """Block until everything enqueued has really happened (a sharded colony may have to repeat passes)."""
        import torch
        if self.world > 1:
            self._confirm(upto=1 << 30)
        torch.cuda.synchronize(self.device)

    def _read_state(self):
        st = _lib.MaacoState.from_buffer_copy(self._state.cpu().numpy().tobytes())
        return st

    def solve_path_planning(self):
        import torch
        K = self.num_iterations
        for it in range(self._iter_done + 1, K + 1):
            self._enqueue_iteration(it)
        self._settle()
        self._iter_done = K
        st = self._read_state()
        # (an explicit max_cells is a limit on the best path even where the sharded exchange grew the buffers)
        limit = self.max_cells if self._auto_cells else self.max_cells_hint
        if st.best_n_cells - 1 > limit:
            if not self._auto_cells or self.max_cells >= self.rows * self.cols:
                raise _lib.MppError(f"a tour outgrew max_cells={limit} (best path: {st.best_n_cells} cells); "
                                    "re-run with a larger max_cells")
            # the solve is a deterministic function of (grid, parameters, seed): repeat it with full path capacity
            again = MAACO(max_cells=self.rows * self.cols, **self._ctor)
            launches = self.kernel_launches + again.kernel_launches
            self.__dict__.update(again.__dict__)
            self.kernel_launches = launches
            return self.solve_path_planning()
        log = self._log.cpu().numpy().reshape(-1, 4)[:K]
        if self.world > 1 and st.best_n_cells > 0:
            import torch.distributed as dist
            owner = st.best_ant // self.n_local                     # rank that constructed the best ant
            dist.broadcast(self._best_cells, src=dist.get_global_rank(self.group, owner), group=self.group)
            torch.cuda.synchronize(self.device)
        cells = self._best_cells[:st.best_n_cells].cpu().numpy()
        self.best_path_overall = [(int(c) // self.cols, int(c) % self.cols) for c in cells]
        self.best_path_length_overall = float(st.best_len)
        self.best_path_turns_overall = int(st.best_turns) if st.best_turns >= 0 else INF
        self.convergence_curve_data = [float(r[2]) if r[2] != INF else None for r in log]  # MAACO.py:360-362
        if self.verbose and self.rank == 0:
            tfmt = lambda v: int(v) if v >= 0 else INF
            for it in range(1, K + 1):                               # MAACO.py:363-366 (printed after the run)
                if it % 10 == 0 or it == 1 or it == K:
                    r = log[it - 1]
                    print(f"MAACO Iter {it}/{K}: Iter Best L={r[0]:.2f}, T={tfmt(r[1])}, "
                          f"Overall Best L={r[2]:.2f}, T={tfmt(r[3])}")
            if self.best_path_overall:
                print(f"\nMAACO Solved: Length={self.best_path_length_overall:.2f}, "
                      f"Turns={self.best_path_turns_overall}")
            else:
                print("\nMAACO: No solution found.")
        return self.best_path_overall, self.best_path_length_overall, self.best_path_turns_overall

    # ---- per-iteration access used by the parity tests and the benchmark -------------------
    def run_iteration(self, it):
        """Enqueue one colony pass; returns nothing (read results with `last_tours`)."""
        self._enqueue_iteration(it)
        self._iter_done = max(self._iter_done, it)

    def run_iteration_host(self, it, tau_in=None, tau_out=None, result_out=None, best_out=None):
        """One colony pass with HOST buffers through the C ABI's mpp_maaco_pass_host (synchronous): `tau_in`
        (rows*cols float64, or None to keep the device field) is copied in, the pass runs, and the updated field, the
        per-ant records (num_ants x {f8 length, i4 n_cells, i4 turns} = 16 bytes each) and the best path so far are
        copied into `tau_out` / `result_out` / `best_out` (NumPy arrays or pinned torch tensors; any may be None).
        Returns the colony state (best length / turns / n_cells ...).  Non-sharded colonies only."""
        import torch
        if self.world != 1:
            raise _lib.MppError("run_iteration_host: a sharded colony exchanges device buffers; use run_iteration")
        if not 1 <= it <= max(1, self.num_iterations):
            raise ValueError(f"iteration {it} outside 1..{self.num_iterations}")

        def hp(x, nbytes):
            if x is None:
                return None
            if isinstance(x, torch.Tensor):
                assert not x.is_cuda and x.is_contiguous() and x.numel() * x.element_size() >= nbytes
                return C.c_void_p(x.data_ptr())
            assert x.flags["C_CONTIGUOUS"] and x.nbytes >= nbytes
            return C.c_void_p(x.ctypes.data)
        n = self.rows * self.cols
        st = _lib.MaacoState()
        cap = 0 if best_out is None else (best_out.numel() if isinstance(best_out, torch.Tensor) else best_out.size)
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(_lib.lib().mpp_maaco_pass_host(
            self._maps, C.byref(self._colony), C.byref(self._params), it, self.num_ants, self._apw, hp(tau_in, n * 8),
            hp(tau_out, n * 8), hp(result_out, self.num_ants * 16), C.byref(st), hp(best_out, 4), cap, stream),
            "mpp_maaco_pass_host")
        self._iter_done = max(self._iter_done, it)
        self.kernel_launches += 4
        return st

    def last_results(self):
        """(n_cells, length, turns) of every ant of the colony in the last pass (numpy).  A colony sharded over peer memory
        receives the other ranks' records from their tour kernels: read them before any rank enqueues the next pass."""
        self._settle()
        raw = self._result.cpu().numpy()
        rec = raw.view(np.dtype([("length", "<f8"), ("n_cells", "<i4"), ("turns", "<i4")])).reshape(-1)
        return rec["n_cells"].copy(), rec["length"].copy(), rec["turns"].copy()

    def last_tours(self):
        """(n_cells, length, turns, cells[n_local, <= max_cells + 1]) of this rank's ants in the last pass; the tours
        are decoded from their move codes (only the columns some tour reached are copied to the host)."""
        nc, ln, tn = self.last_results()
        sl = slice(self.ant_offset, self.ant_offset + self.n_local)
        used = int(min(self.max_cells, max(1, nc[sl].max(initial=1) - 1)))
        mv = self._moves.view(self.n_local, self.max_cells)[:, :used].cpu().numpy()
        dr = np.array([-1, -1, -1, 0, 0, 1, 1, 1])                     # move order MAACO.py:98
        dc = np.array([-1, 0, 1, -1, 1, -1, 0, 1])
        delta = (dr * self.cols + dc).astype(np.int64)[mv & 7]
        cells = np.empty((self.n_local, used + 1), np.int64)
        cells[:, 0] = self.start_node[0] * self.cols + self.start_node[1]
        np.cumsum(delta, axis=1, out=cells[:, 1:])
        cells[:, 1:] += cells[:, :1]
        return nc[sl], ln[sl], tn[sl], cells.astype(np.int32)

    def total_steps(self):
        self._settle()
        return int(self._steps.cpu().item())

    # ---- plotting hooks of the reference (MAACO.py:373-377): out of scope, forwarded if possible --
    def visualize_pheromone_matrix(self, title="Mức Pheromone MAACO"):
        try:
            from visualization import visualize_pheromone_matrix as viz
        except Exception:
            print("visualization/matplotlib not available; pheromone_matrix is exposed as an ndarray")
            return
        viz(self.grid, self.pheromone_matrix, title)

    def plot_convergence_curve(self):
        try:
            from visualization import plot_convergence_curve as viz
        except Exception:
            print("visualization/matplotlib not available; convergence_curve_data is exposed as a list")
            return
        viz(self.convergence_curve_data, "MAACO", color='orangered')
